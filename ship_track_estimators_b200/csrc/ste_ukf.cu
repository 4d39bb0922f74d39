// ste_ukf.cu - kernels and C ABI of libste_ukf.so (sm_100a only).
//
// Execution model: one thread per track, sequential in time (the UKF recursion is a
// loop-carried dependency through sqrtm + trigonometry; tracks are the parallel axis).
// All arrays are [plane][track] so that a warp's 32 loads/stores of one plane are one
// contiguous 256-byte segment.  The kernels are bound by the FP64 pipe (about 26 flop per
// algorithmic byte, DESIGN.md), so the time loop keeps every matrix in registers and
// prefetches the next step's inputs while the current step computes.
#include <cmath>
#include <cstdio>
#include <cstring>

#include "ste_tracks.cuh"
#include "ste_generic.cuh"
#include "ste_ingest.cuh"

namespace ste {

#ifndef STE_THREADS
#define STE_THREADS 128
#endif
constexpr int kThreads = STE_THREADS;
// Minimum resident blocks per SM the register allocator must make room for (measured optima):
//  - forward: 3 blocks = 12 warps at 159 registers, no spills (2 blocks: -5 %, 4 blocks: spills);
//  - backward over the statistics tape: HBM-bound, and what hurts it is local-memory traffic, so
//    it gets the registers it asks for (227, no spills) at 2 blocks = 8 warps: 13.7e9 track-steps/s
//    against 10.2e9 at 4 blocks / 128 registers / 208 B of spills;
//  - backward by recomputation (no tape): compute-bound like the forward pass, 3 blocks (shared memory).
#ifndef STE_FWD_MIN_BLOCKS
#define STE_FWD_MIN_BLOCKS 3
#endif
#ifndef STE_BWD_MIN_BLOCKS
#define STE_BWD_MIN_BLOCKS 2
#endif
#ifndef STE_BWD_RECOMPUTE_MIN_BLOCKS
#define STE_BWD_RECOMPUTE_MIN_BLOCKS 3   // 62 scratch slots per thread: three 62 KB blocks per SM
#endif

// INNOV: the launch also writes the innovation statistics of every update.  Their planes travel in a parameter block of
// their own (KernelArgsInnov), so that KernelArgs - and with it every other kernel's parameters - stays as it was.
struct KernelArgsInnov : KernelArgs {
    SteInnovations innov;
};
// PER_Q: every track has its own process noise (ste_ukf_forward_noise_f64 / ste_urtss_backward_noise_f64).  The plane
// pointer travels in a parameter block read only by the PER_Q instantiations, after everything the others read; `innov`
// is read only by the forward instantiations that write the statistics.
struct KernelArgsQ : KernelArgsInnov {
    const double *Q_tracks;   // [16][ld] row-major per-track Q
};
template <bool INNOV, bool PER_Q = false> struct ForwardArgs { using type = KernelArgs; };
template <> struct ForwardArgs<true> { using type = KernelArgsInnov; };
template <bool INNOV> struct ForwardArgs<INNOV, true> { using type = KernelArgsQ; };

template <bool POS_ONLY, bool GATING, bool INNOV = false, bool PER_Q = false>
__global__ void __launch_bounds__(kThreads, STE_FWD_MIN_BLOCKS) ukf_forward_kernel(const __grid_constant__ typename ForwardArgs<INNOV, PER_Q>::type a) {
    extern __shared__ double scratch[];   // kScratchSlotsFwd * kThreads doubles (62 KB: opt-in size)
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if constexpr (PER_Q) {
        if (t < a.prob.n_tracks)
            forward_track<POS_ONLY, GATING, INNOV, false, true>(a, t, Scratch{scratch + threadIdx.x, kThreads}, INNOV ? &a.innov : nullptr,
                                                                nullptr, 0, a.Q_tracks);
    } else if constexpr (INNOV) {
        if (t < a.prob.n_tracks) forward_track<POS_ONLY, GATING, true>(a, t, Scratch{scratch + threadIdx.x, kThreads}, &a.innov);
    } else {
        if (t < a.prob.n_tracks) forward_track<POS_ONLY, GATING>(a, t, Scratch{scratch + threadIdx.x, kThreads});
    }
}

// Scoring form of the forward pass (ste_ukf_score_f64): blockIdx.y is the candidate, so every warp reads one candidate's
// Q and R from the parameter block.  Each (candidate, track) pair runs forward_track's arithmetic with the candidate's
// matrices and writes only its sums.
template <bool POS_ONLY, bool GATING>
__global__ void __launch_bounds__(kThreads, STE_FWD_MIN_BLOCKS) ukf_score_kernel(const __grid_constant__ KernelArgsScore a) {
    extern __shared__ double scratch[];   // kScratchSlotsFwd * kThreads doubles, as the forward pass
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < a.prob.n_tracks) forward_track<POS_ONLY, GATING, false, true>(a, t, Scratch{scratch + threadIdx.x, kThreads}, nullptr, &a, blockIdx.y);
}

// TAPE: the launch has a statistics tape (same code either way; only the register budget differs).  PER_Q: as the forward.
template <bool TAPE, bool PER_Q = false>
__global__ void __launch_bounds__(kThreads, TAPE ? STE_BWD_MIN_BLOCKS : STE_BWD_RECOMPUTE_MIN_BLOCKS)
urtss_backward_kernel(const __grid_constant__ typename ForwardArgs<false, PER_Q>::type a) {
    extern __shared__ double scratch[];   // kScratchSlotsBwd * kThreads doubles (46 KB: opt-in size)
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if constexpr (PER_Q) {
        if (t < a.prob.n_tracks) backward_track<true>(a, t, Scratch{scratch + threadIdx.x, kThreads}, a.Q_tracks);
    } else {
        if (t < a.prob.n_tracks) backward_track(a, t, Scratch{scratch + threadIdx.x, kThreads});
    }
}

// Co-resident passes: ONE launch whose blocks take one of two roles - forward filter of tile a or backward smoother
// of tile b (already filtered, statistics on its tape).  The filter is bound by the FP64 pipe and leaves DRAM idle, the
// tape smoother is bound by DRAM and leaves the FP64 pipe idle; run back to back their times add.  Here the roles are
// interleaved along blockIdx in proportion to the two block counts, so that every SM holds both kinds at once (the block
// scheduler hands out blocks in index order, and the quicker smoother blocks turn over faster, which settles the
// resident mix by itself) and the smoother's memory round trips pass behind the filter's arithmetic.  Every track runs
// exactly the code of the separate kernels: results are bit-identical to forward(a) then backward(b).
#ifndef STE_ROLES_MIN_BLOCKS
#define STE_ROLES_MIN_BLOCKS 3   // both roles within 168 registers: any three blocks fit one SM
#endif
struct RoleSplit {
    int blocks_a, blocks_b;   // forward blocks (tile a), backward blocks (tile b)
};
template <bool POS_ONLY, bool GATING>
__global__ void __launch_bounds__(kThreads, STE_ROLES_MIN_BLOCKS)
ukf_roles_kernel(const __grid_constant__ KernelArgs a, const __grid_constant__ KernelArgs b, const RoleSplit split) {
    extern __shared__ double scratch[];   // kScratchSlots * kThreads doubles (either role)
    // block i is a forward block when floor((i + 1) * A / N) > floor(i * A / N): A of N blocks, evenly spread
    const long long A = split.blocks_a, N = (long long)split.blocks_a + split.blocks_b, i = blockIdx.x;
    const int fa = (int)(i * A / N), fa1 = (int)((i + 1) * A / N);
    const Scratch sc{scratch + threadIdx.x, kThreads};
    if (fa1 > fa) {
        const int t = fa * kThreads + threadIdx.x;
        if (t < a.prob.n_tracks) forward_track<POS_ONLY, GATING>(a, t, sc);
    } else {
        const int t = ((int)i - fa) * kThreads + threadIdx.x;
        if (t < b.prob.n_tracks) backward_track(b, t, sc);
    }
}

// ------------------------------------------------------------------------------------------ //
// Single-step entry points behind UnscentedKalmanFilter.predict / .update.
// ------------------------------------------------------------------------------------------ //
struct StepArgs {
    SteProblem prob;
    double *x;
    double *P;
    const double *dt, *sog_rate, *cog_rate, *noise, *z;
    double *sigma_prior, *sigma_post;
    uint8_t *gate_iters;
    double *gate_lambda;
    double *gate_scale;
    int32_t *status;
};

__device__ __forceinline__ void load_xP(const StepArgs &a, int t, double (&x)[4], double (&P)[10]) {
    const int64_t ld = a.prob.ld;
#pragma unroll
    for (int r = 0; r < 4; ++r) x[r] = a.x[r * ld + t];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) P[SYM(i, j)] = a.P[(i * 4 + j) * ld + t];
}
__device__ __forceinline__ void store_xP(const StepArgs &a, int t, const double (&x)[4], const double (&P)[10]) {
    const int64_t ld = a.prob.ld;
#pragma unroll
    for (int r = 0; r < 4; ++r) a.x[r * ld + t] = x[r];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) a.P[(i * 4 + j) * ld + t] = P[SYM(i, j)];
}

constexpr int kStepThreads = 64;   // single-step predict: 62 scratch slots per thread within the static 48 KB
__global__ void __launch_bounds__(kStepThreads) ukf_predict_kernel(const __grid_constant__ StepArgs a) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.prob.n_tracks) return;
    const int64_t ld = a.prob.ld;
    double x[4], P[10], e[4] = {0.0, 0.0, 0.0, 0.0};
    load_xP(a, t, x, P);
    if (a.noise) {
#pragma unroll
        for (int r = 0; r < 4; ++r) e[r] = a.noise[r * ld + t] * sqrt(a.prob.Q[r * 5]);
    }
    int status = 0;
    __shared__ double scratch[kScratchSlots * kStepThreads];
    ukf_predict(x, P, a.prob.Q, a.dt[t], a.sog_rate[t], a.cog_rate[t], e, status, Scratch{scratch + threadIdx.x, kStepThreads},
                a.sigma_prior ? a.sigma_prior + t : nullptr, a.sigma_post ? a.sigma_post + t : nullptr, nullptr, ld,
                !(a.prob.flags & STE_FLAG_LONG_STEPS));
    if (any_nonfinite(x, P)) status |= STE_STATUS_NONFINITE;
    store_xP(a, t, x, P);
    if (a.status) a.status[t] = status;
}

template <bool POS_ONLY, bool GATING>
__global__ void __launch_bounds__(kThreads) ukf_update_kernel(const __grid_constant__ StepArgs a) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.prob.n_tracks) return;
    const int64_t ld = a.prob.ld;
    const Model model{a.prob.H, a.prob.Q, a.prob.R};
    double x[4], P[10], z[4], un[4];
    load_xP(a, t, x, P);
#pragma unroll
    for (int r = 0; r < 4; ++r) z[r] = a.z[r * ld + t];
    const double *noise = nullptr;
    if (a.noise) {
#pragma unroll
        for (int r = 0; r < 4; ++r) un[r] = a.noise[r * ld + t];
        noise = un;
    }
    int status = 0, it;
    double lam, rs;
    if (POS_ONLY)
        ukf_update_position<GATING>(x, P, model, z, noise, a.prob.gate_chi, a.prob.gate_max_iter, status, it, lam, rs);
    else
        ukf_update_generic<GATING>(x, P, model, z, noise, a.prob.gate_chi, a.prob.gate_max_iter, status, it, lam, rs);
    if (any_nonfinite(x, P)) status |= STE_STATUS_NONFINITE;
    store_xP(a, t, x, P);
    if (a.gate_iters) a.gate_iters[t] = (uint8_t)min_(it, 255);
    if (a.gate_lambda) a.gate_lambda[t] = lam;
    if (a.gate_scale) a.gate_scale[t] = rs;
    if (a.status) a.status[t] = status;
}

// criterion_index / update_lambda_factor (unscented.py:389-483): gamma = |y^T S^+ y| and the
// denominator y^T S^+ R S^+ y of the lambda update, y = z - x (not z - Hx, no wrap), S = H P H^T + R.
__global__ void __launch_bounds__(kThreads) gate_terms_kernel(const __grid_constant__ StepArgs a, double *gamma, double *denom) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.prob.n_tracks) return;
    const int64_t ld = a.prob.ld;
    double x[4], P[10], y[4], HP[16], S[10], Sinv[10], v[4];
    load_xP(a, t, x, P);
#pragma unroll
    for (int r = 0; r < 4; ++r) y[r] = a.z[r * ld + t] - x[r];
    innovation_cov(P, a.prob.H, a.prob.R, 1.0, HP, S);
    pinv_sym4(S, Sinv);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double acc = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) acc = fma(Sinv[SYM(i, j)], y[j], acc);
        v[i] = acc;
    }
    double den = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double row = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) row = fma(a.prob.R[i * 4 + j], v[j], row);
        den = fma(v[i], row, den);
    }
    gamma[t] = fabs(quad_form(Sinv, y));
    denom[t] = den;
}

// ------------------------------------------------------------------------------------------ //
// compute_sigma_points for any n <= 8 (unscented.py:76-107).  Not on the hot path: generic-n
// cyclic Jacobi on thread-local arrays.
// ------------------------------------------------------------------------------------------ //
__global__ void __launch_bounds__(kThreads) sigma_points_kernel(int n, int T, int64_t ld, double scale, const double *x,
                                                                 const double *P, double *X, int32_t *status) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    double A[64], V[64];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) {
            // the root is taken of the symmetric part; P is symmetric up to rounding in the filter
            A[i * 8 + j] = 0.5 * scale * (P[(i * n + j) * ld + t] + P[(j * n + i) * ld + t]);
            V[i * 8 + j] = (i == j) ? 1.0 : 0.0;
        }
    for (int sweep = 0; sweep < 30; ++sweep) {
        double off = 0.0, dia = 0.0;
        for (int i = 0; i < n; ++i) {
            dia += A[i * 8 + i] * A[i * 8 + i];
            for (int j = i + 1; j < n; ++j) off += A[i * 8 + j] * A[i * 8 + j];
        }
        if (!(off > 1e-36 * dia)) break;
        for (int p = 0; p < n - 1; ++p)
            for (int q = p + 1; q < n; ++q) {
                const double apq = A[p * 8 + q];
                if (apq == 0.0) continue;
                const double d = A[q * 8 + q] - A[p * 8 + p], b = apq + apq;
                const double tt = (d >= 0.0 ? b : -b) / (fabs(d) + sqrt(fma(d, d, b * b)));
                const double c = fast_rsqrt(fma(tt, tt, 1.0)), s = tt * c;
                for (int r = 0; r < n; ++r) {  // columns p, q of A and V
                    const double arp = A[r * 8 + p], arq = A[r * 8 + q];
                    A[r * 8 + p] = fma(c, arp, -s * arq);
                    A[r * 8 + q] = fma(s, arp, c * arq);
                    const double vrp = V[r * 8 + p], vrq = V[r * 8 + q];
                    V[r * 8 + p] = fma(c, vrp, -s * vrq);
                    V[r * 8 + q] = fma(s, vrp, c * vrq);
                }
                for (int r = 0; r < n; ++r) {  // rows p, q of A
                    const double apr = A[p * 8 + r], aqr = A[q * 8 + r];
                    A[p * 8 + r] = fma(c, apr, -s * aqr);
                    A[q * 8 + r] = fma(s, apr, c * aqr);
                }
                A[p * 8 + q] = 0.0;
                A[q * 8 + p] = 0.0;
            }
    }
    int st = 0;
    double wmax = 0.0;
    for (int k = 0; k < n; ++k) wmax = fmax(wmax, fabs(A[k * 8 + k]));
    double f[8];
    for (int k = 0; k < n; ++k) {
        if (A[k * 8 + k] < -1e-13 * wmax) st |= STE_STATUS_INDEFINITE;
        f[k] = sqrt(fmax(A[k * 8 + k], 0.0));
    }
    const int L = 2 * n + 1;
    for (int r = 0; r < n; ++r) {
        const double xr = x[r * ld + t];
        X[(r * L) * ld + t] = xr;
        for (int i = 0; i < n; ++i) {
            double m = 0.0;
            for (int k = 0; k < n; ++k) m = fma(V[r * 8 + k] * f[k], V[i * 8 + k], m);
            X[(r * L + 1 + i) * ld + t] = xr + m;
            X[(r * L + 1 + n + i) * ld + t] = xr - m;
        }
    }
    if (status) status[t] = st;
}

__global__ void __launch_bounds__(kThreads) geodetic_kernel(int T, int64_t ld, const double *xin, const double *dt,
                                                            const double *sog_rate, const double *cog_rate,
                                                            double *xout) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    double x[4], y[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) x[r] = xin[r * ld + t];
    const double d = dt[t];
    geodetic_step(x, d, d / kEarthRadiusKm, sog_rate[t], cog_rate[t], y);
#pragma unroll
    for (int r = 0; r < 4; ++r) xout[r * ld + t] = y[r];
}

// ------------------------------------------------------------------------------------------ //
// performance_metrics.py:4-58 over whole tiles: residuals between a state estimate and the
// observations it assimilated, one thread per track walking the forward pass's update cadence.
// Streaming reads of [step][row][track] planes; HBM-bound (two to four doubles per update).
// ------------------------------------------------------------------------------------------ //
// NS = 4 reads the n = 4 tile (SteProblem / SteInputs, cadence from upd_mask or substeps), NS = 5 the five-state fleet
// tile (SteProblemN / SteInputsN, upd_mask required).  The arithmetic is the same for both.
template <int NS> struct MetricsTile;
template <> struct MetricsTile<4> {
    using Problem = SteProblem;
    using Inputs = SteInputs;
    __device__ static int substeps(const SteProblem &p) { return p.substeps > 0 ? p.substeps : 1; }
};
template <> struct MetricsTile<5> {
    using Problem = SteProblemN;
    using Inputs = SteInputsN;
    __device__ static int substeps(const SteProblemN &) { return 1; }
};

template <int NS>
struct MetricsArgs {
    typename MetricsTile<NS>::Problem prob;
    typename MetricsTile<NS>::Inputs in;
    const double *mean;
    double *rmse, *cum_abs, *max_abs, *abs_diff;
    int32_t *n_pairs;
};

// One thread per (track, observation row): the rows of a track are independent sums, and twice (position-only) to four
// times the threads of a one-thread-per-track launch keep twice to four times the loads in flight.  blockIdx.y
// counts the rows that exist (z[r] != NULL), in order.
template <int NS>
__global__ void __launch_bounds__(kThreads) track_metrics_kernel(const __grid_constant__ MetricsArgs<NS> a) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.prob.n_tracks) return;
    int r = 0;
    for (int seen = -1; r < NS; ++r) {
        if (a.in.z[r] && ++seen == (int)blockIdx.y) break;
    }
    const int64_t ld = a.prob.ld;
    const int nt = a.in.n_steps ? min(a.in.n_steps[t], a.prob.max_steps) : a.prob.max_steps;
    const int k_sub = MetricsTile<NS>::substeps(a.prob);
    const double *zr = a.in.z[r] + t;
    const double *mr = a.mean + (int64_t)r * ld + t;
    double sq = 0.0, sa = 0.0, mx = 0.0;
    int pairs = 0, ui = 0;
    auto pair = [&](int state, int obs) {
        const double d = fabs(STE_LOAD_STREAM(mr + ((int64_t)state * NS) * ld) - zr[(int64_t)obs * ld]);
        sq = fma(d, d, sq);
        sa += d;
        mx = fmax(mx, d);   // NaN residuals propagate through sq / sa
        if (a.abs_diff) STE_STORE_STREAM(a.abs_diff + ((int64_t)obs * NS + r) * ld + t, d);
        ++pairs;
    };
    pair(0, 0);
    // (unrolling this loop so that several steps' loads are in flight was measured slower: 1.19 ms
    // against 0.71 ms for 113 664 x 512 - consecutive steps are megabytes apart)
    for (int s = 0; s < nt; ++s) {
        const bool upd = a.in.upd_mask ? (a.in.upd_mask[(int64_t)s * ld + t] != 0) : ((s + 1) % k_sub == 0);
        if (upd && ui + 1 < a.prob.max_obs) pair(s + 1, ++ui);
    }
    if (a.rmse) a.rmse[r * ld + t] = sqrt(sq / (double)pairs);
    if (a.cum_abs) a.cum_abs[r * ld + t] = sa;
    if (a.max_abs) a.max_abs[r * ld + t] = mx;
    if (a.n_pairs && blockIdx.y == 0) a.n_pairs[t] = pairs;
}

// ------------------------------------------------------------------------------------------ //
// Derived filter inputs from raw fixes (SURVEY section 8(f) row N1): what ShipTrack computes per
// ship on the host (ship_track.py:197-304) with the spherical pair haversine_formula / heading
// (utils.py:75-147), plus the CLI's optional box smoothing of SOG and COG (utils.py:150-172,
// main_cli.py:99-104).  One thread per track, sequential over its fixes; not a hot path, so the
// CUDA math library is used as is.  The rate arrays double as scratch for the unsmoothed values.
// ------------------------------------------------------------------------------------------ //
__device__ __forceinline__ void leg_speed_course(double lon1, double lat1, double lon2, double lat2, double dt,
                                                 double &sog, double &cog) {
    const double l1 = lon1 * kDegToRad, p1 = lat1 * kDegToRad, l2 = lon2 * kDegToRad, p2 = lat2 * kDegToRad;
    const double dphi = p2 - p1, dlam = l2 - l1;
    const double sh = sin(dphi / 2.0), sl = sin(dlam / 2.0);
    const double cp1 = cos(p1), cp2 = cos(p2);
    const double a = sh * sh + cp1 * cp2 * (sl * sl);
    const double dist = (2.0 * atan2(sqrt(a), sqrt(1.0 - a))) * kEarthRadiusKm;   // utils.py:104-111
    sog = dist / dt;                                                                 // ship_track.py:213-217
    const double east = sin(dlam) * cp2;
    const double north = cp1 * sin(p2) - sin(p1) * cp2 * cos(dlam);
    cog = py_mod360(atan2(east, north) * kRadToDeg + 360.0);                       // utils.py:139-145
}

// WGS84 leg: Vincenty's inverse formulae (Survey Review 23 (176), 1975) for the distance s12 and the
// initial azimuth the reference takes from geographiclib (utils.py:36-37, 68-70).
__device__ __forceinline__ void leg_speed_course_wgs84(double lon1, double lat1, double lon2, double lat2, double dt,
                                                       double &sog, double &cog) {
    if (fabs(lat1 - lat2) < 1e-8 && fabs(lon1 - lon2) < 1e-8) {   // utils.py:32-33, 64-65
        sog = 0.0 / dt;
        cog = 0.0;
        return;
    }
    constexpr double a = 6378137.0, f = 1.0 / 298.257223563, b = (1.0 - f) * a;
    const double U1 = atan((1.0 - f) * tan(lat1 * kDegToRad)), U2 = atan((1.0 - f) * tan(lat2 * kDegToRad));
    const double L = (lon2 - lon1) * kDegToRad;
    const double sU1 = sin(U1), cU1 = cos(U1), sU2 = sin(U2), cU2 = cos(U2);
    double lam = L, sl, cl, ss, cs, sig, sa, c2a, c2sm;
    bool converged = false;
    for (int it = 0; it < 200; ++it) {
        sl = sin(lam); cl = cos(lam);
        ss = hypot(cU2 * sl, cU1 * sU2 - sU1 * cU2 * cl);
        cs = sU1 * sU2 + cU1 * cU2 * cl;
        sig = atan2(ss, cs);
        sa = cU1 * cU2 * sl / ss;
        c2a = 1.0 - sa * sa;
        c2sm = c2a != 0.0 ? cs - 2.0 * sU1 * sU2 / c2a : 0.0;
        const double C = f / 16.0 * c2a * (4.0 + f * (4.0 - 3.0 * c2a));
        const double next = L + (1.0 - C) * f * sa * (sig + C * ss * (c2sm + C * cs * (-1.0 + 2.0 * c2sm * c2sm)));
        const double d = fabs(next - lam);
        lam = next;
        if (d < 1e-15) { converged = true; break; }
    }
    sl = sin(lam); cl = cos(lam);
    const double ty = cU2 * sl, tx = cU1 * sU2 - sU1 * cU2 * cl;
    ss = hypot(ty, tx);
    cs = sU1 * sU2 + cU1 * cU2 * cl;
    sig = atan2(ss, cs);
    sa = cU1 * cU2 * sl / ss;
    c2a = 1.0 - sa * sa;
    c2sm = c2a != 0.0 ? cs - 2.0 * sU1 * sU2 / c2a : 0.0;
    const double u2 = c2a * (a * a - b * b) / (b * b);
    const double A = 1.0 + u2 / 16384.0 * (4096.0 + u2 * (-768.0 + u2 * (320.0 - 175.0 * u2)));
    const double B = u2 / 1024.0 * (256.0 + u2 * (-128.0 + u2 * (74.0 - 47.0 * u2)));
    const double dsig = B * ss * (c2sm + B / 4.0 * (cs * (-1.0 + 2.0 * c2sm * c2sm)
                                                   - B / 6.0 * c2sm * (-3.0 + 4.0 * ss * ss) * (-3.0 + 4.0 * c2sm * c2sm)));
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    const double s12 = converged ? b * A * (sig - dsig) : nan;
    sog = (s12 * 1e-3) / dt;                                                   // utils.py:37, ship_track.py:213-217
    cog = converged ? py_mod360(atan2(ty, tx) * kRadToDeg + 360.0) : nan;       // utils.py:69-70
}

__global__ void __launch_bounds__(kThreads) derive_inputs_kernel(int T, int max_obs, int64_t ld, int width, int geodesy,
                                                                 const double *lon, const double *lat, const double *dts,
                                                                 const int32_t *n_obs, double *sog, double *cog,
                                                                 double *sog_rate, double *cog_rate) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int n = n_obs ? min(n_obs[t], max_obs) : max_obs;
    const bool smoothing = width > 1;
    double *raw_s = smoothing ? sog_rate : sog, *raw_c = smoothing ? cog_rate : cog;
    auto at = [&](const double *p, int i) { return p[(int64_t)i * ld + t]; };
    auto put = [&](double *p, int i, double v) { p[(int64_t)i * ld + t] = v; };
    // pass 1: one value per leg, the last one repeated ("stationary from the end point onwards")
    double s = 0.0, c = 0.0;
    for (int i = 0; i + 1 < n; ++i) {
        if (geodesy == STE_GEODESY_WGS84) leg_speed_course_wgs84(at(lon, i), at(lat, i), at(lon, i + 1), at(lat, i + 1), at(dts, i), s, c);
        else leg_speed_course(at(lon, i), at(lat, i), at(lon, i + 1), at(lat, i + 1), at(dts, i), s, c);
        put(raw_s, i, s);
        put(raw_c, i, c);
    }
    if (n > 0) {
        put(raw_s, n - 1, s);
        put(raw_c, n - 1, c);
    }
    // pass 2: np.convolve(y, ones(w) / w, mode="same") with zero padding: out[i] = sum_tap y[i + start - tap] / w
    if (smoothing) {
        const int start = (width - 1) / 2;
        const double inv_w = 1.0 / (double)width;
        for (int i = 0; i < n; ++i) {
            double as = 0.0, ac = 0.0;
            for (int tap = width - 1; tap >= 0; --tap) {
                const int j = i + start - tap;
                if (j >= 0 && j < n) {
                    as = fma(at(raw_s, j), inv_w, as);
                    ac = fma(at(raw_c, j), inv_w, ac);
                }
            }
            put(sog, i, as);
            put(cog, i, ac);
        }
    }
    // pass 3: backward differences with a leading zero (ship_track.py:242-248, 296-302)
    double ps = n > 0 ? at(sog, 0) : 0.0, pc = n > 0 ? at(cog, 0) : 0.0;
    if (n > 0) {
        put(sog_rate, 0, 0.0);
        put(cog_rate, 0, 0.0);
    }
    for (int i = 1; i < n; ++i) {
        const double vs = at(sog, i), vc = at(cog, i), d = at(dts, i - 1);
        put(sog_rate, i, (vs - ps) / d);
        put(cog_rate, i, (vc - pc) / d);
        ps = vs;
        pc = vc;
    }
    for (int i = n; i < max_obs; ++i) {   // padding rows of ragged tiles
        put(sog, i, 0.0);
        put(cog, i, 0.0);
        put(sog_rate, i, 0.0);
        put(cog_rate, i, 0.0);
    }
}

// ------------------------------------------------------------------------------------------ //
// Dimension-generic single steps (ste_generic.cuh): the class API for n != 4 / other process models.
// ------------------------------------------------------------------------------------------ //
__global__ void __launch_bounds__(64) ukf_predict_n_kernel(const __grid_constant__ ProblemN p, double *x, double *P, const double *dt,
                                                            const double *sog_rate, const double *cog_rate, const double *noise,
                                                            double *sigma_prior, double *sigma_post, int32_t *status) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < p.n_tracks) predict_n(p, t, x, P, dt, sog_rate, cog_rate, noise, sigma_prior, sigma_post, status);
}

__global__ void __launch_bounds__(64) ukf_update_n_kernel(const __grid_constant__ ProblemN p, double *x, double *P, const double *z,
                                                           const double *noise, int32_t *status) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < p.n_tracks) update_n(p, t, x, P, z, noise, status);
}

__global__ void __launch_bounds__(64) urtss_backward_n_kernel(const __grid_constant__ ProblemN p, int n_states, int rate_repeat, int n_rates,
                                                             const double *mean_f, const double *cov_f, const double *dt,
                                                             const double *sog_rate, const double *cog_rate, const double *noise,
                                                             double *mean_s, double *cov_s, int32_t *status) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.n_tracks) return;
    const int st = rts_n<0>(p, p.Q, t, n_states, rate_repeat, n_rates, mean_f, cov_f, dt, sog_rate, cog_rate, noise, mean_s, cov_s);
    if (status) status[t] = st;
}

// ------------------------------------------------------------------------------------------ //
// Whole-track fleet kernels at a compile-time dimension (NC = 5: geodetic_dynamics_turn).  One thread
// per track, the state thread-local across the time loop; the arithmetic is the single-step kernels'
// (predict_core / update_core / rts_n of ste_generic.cuh), so every track is bit-identical to the
// class API's step-by-step route.
// ------------------------------------------------------------------------------------------ //
#ifndef STE_N5_THREADS
#define STE_N5_THREADS 64
#endif
constexpr int kThreadsN = STE_N5_THREADS;

struct FleetArgsN {
    ProblemN p;
    double P0[kMaxN * kMaxN];   // shared prior, row-major n x n
    int32_t max_steps, max_obs;
    SteInputsN in;
    SteOutputsN out;
    SteNoiseN noise;   // per-track Q / R planes, or NULL (last, so the shared path's parameter offsets stay as they were)
    SteInnovations innov;   // innovation statistics planes (read by the Innov instantiation only)
};

// Q and R of track t: with PerTrack, its own planes (noise.Q_tracks / R_tracks, the launch's matrix where one is NULL)
// loaded once, before the time loop; otherwise the launch's matrices, read from the kernel parameters.  The host picks
// PerTrack only when a plane set is present, so a launch without one keeps the shared path's code and registers.
template <int NC, bool PerTrack>
STE_DEV const double *track_matrix(const double *shared, const double *planes, int64_t ld, int t, double *own) {
    if constexpr (PerTrack) {
        for (int k = 0; k < NC * NC; ++k) own[k] = planes ? planes[k * ld + t] : shared[k];
        return own;
    } else {
        return shared;
    }
}

// KalmanFilterBase.run (kalman_filter.py:36-117): row 0 the prior, the initial update with observation 0, then per step
// a predict with the rates of the current update index and, where upd_mask is set, an update with the next observation.
// Innov: every update also stores its innovation statistics into row u of a.innov's planes.
template <int NC, bool PerTrack, bool Innov = false>
__global__ void __launch_bounds__(kThreadsN) ukf_forward_n_kernel(const __grid_constant__ FleetArgsN a) {
    constexpr int D = DimN<NC>::LD, n = NC;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.p.n_tracks) return;
    const SteInputsN &in = a.in;
    const int64_t ld = a.p.ld;
    const int nt = in.n_steps ? min(in.n_steps[t], a.max_steps) : a.max_steps;
    double x[D], P[D * D], z[D], Qt[PerTrack ? n * n : 1], Rt[PerTrack ? n * n : 1];
    const double *Q = track_matrix<NC, PerTrack>(a.p.Q, a.noise.Q_tracks, ld, t, Qt);
    const double *R = track_matrix<NC, PerTrack>(a.p.R, a.noise.R_tracks, ld, t, Rt);
    for (int r = 0; r < n; ++r) x[r] = in.x0[r * ld + t];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) P[i * D + j] = in.P0 ? in.P0[(i * n + j) * ld + t] : a.P0[i * n + j];
    auto store = [&](int s) {
        for (int r = 0; r < n; ++r) {
            a.out.mean_f[((int64_t)s * n + r) * ld + t] = x[r];
            for (int q = 0; q < n; ++q) a.out.cov_f[((int64_t)s * n * n + r * n + q) * ld + t] = P[r * D + q];
        }
    };
    auto update = [&](int u) {   // observation row u; rows the caller left NULL read as 0
        for (int r = 0; r < n; ++r) z[r] = in.z[r] ? in.z[r][(int64_t)u * ld + t] : 0.0;
        if constexpr (Innov) {
            ste::Innov st;
            const int bits = update_core<NC, true>(a.p, R, x, P, z, in.noise_upd ? in.noise_upd + (int64_t)u * n * ld + t : nullptr, ld, &st);
            const int64_t row = (int64_t)u * ld + t;
            a.innov.nis[row] = st.nis;
            a.innov.loglik[row] = -0.5 * fma((double)st.rank, kLog2Pi, st.nis + st.log_pdet);
            a.innov.rank[row] = (uint8_t)st.rank;
            return bits;
        } else {
            return update_core<NC>(a.p, R, x, P, z, in.noise_upd ? in.noise_upd + (int64_t)u * n * ld + t : nullptr, ld);
        }
    };
    store(0);                      // :76-81
    int status = update(0), ui = 0;
    for (int s = 0; s < nt; ++s) {
        const double d = in.dt[(int64_t)s * ld + t], sr = in.sog_rate[(int64_t)ui * ld + t],
                     cr = in.cog_rate ? in.cog_rate[(int64_t)ui * ld + t] : 0.0;
        status |= predict_core<NC>(a.p, Q, x, P, d, sr, cr, in.noise_pred ? in.noise_pred + (int64_t)s * n * ld + t : nullptr, ld,
                                   nullptr, nullptr, 0);
        if (in.upd_mask[(int64_t)s * ld + t]) {   // :101-108
            if (ui + 1 < a.max_obs) status |= update(++ui);
            else status |= STE_STATUS_OBS_OVERRUN;
        }
        store(s + 1);
    }
    a.out.status[t] = status;
    if (a.out.n_updates) a.out.n_updates[t] = ui + 1;
}

// Scoring form of ukf_forward_n_kernel (ste_ukf_score_n_f64): the same time loop, predict_core / update_core calls and
// statistics, with the Q and R of candidate blockIdx.y (so every warp reads one candidate's matrices) and no stored state;
// the statistics of the updates are summed in update order and written once per (candidate, track).
struct ScoreArgsN {
    ProblemN p;
    double P0[kMaxN * kMaxN];   // shared prior, row-major n x n
    int32_t max_steps, max_obs;
    SteInputsN in;
    SteScores scores;
    double Q[STE_MAX_CANDIDATES][25], R[STE_MAX_CANDIDATES][25];   // row-major n x n per candidate
};

template <int NC>
__global__ void __launch_bounds__(kThreadsN) ukf_score_n_kernel(const __grid_constant__ ScoreArgsN a) {
    static_assert(NC * NC <= 25, "the candidate table holds 5 x 5 matrices");
    constexpr int D = DimN<NC>::LD, n = NC;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.p.n_tracks) return;
    const int c = blockIdx.y;
    const SteInputsN &in = a.in;
    const int64_t ld = a.p.ld;
    const int nt = in.n_steps ? min(in.n_steps[t], a.max_steps) : a.max_steps;
    const double *Q = a.Q[c], *R = a.R[c];
    double x[D], P[D * D], z[D];
    for (int r = 0; r < n; ++r) x[r] = in.x0[r * ld + t];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) P[i * D + j] = in.P0 ? in.P0[(i * n + j) * ld + t] : a.P0[i * n + j];
    double loglik = 0.0, nis = 0.0;
    int dof = 0;
    auto update = [&](int u) {   // observation row u; rows the caller left NULL read as 0
        for (int r = 0; r < n; ++r) z[r] = in.z[r] ? in.z[r][(int64_t)u * ld + t] : 0.0;
        ste::Innov st;
        const int bits = update_core<NC, true>(a.p, R, x, P, z, in.noise_upd ? in.noise_upd + (int64_t)u * n * ld + t : nullptr, ld, &st);
        loglik += -0.5 * fma((double)st.rank, kLog2Pi, st.nis + st.log_pdet);   // the loglik plane's expression
        nis += st.nis;
        dof += st.rank;
        return bits;
    };
    int status = update(0), ui = 0;
    for (int s = 0; s < nt; ++s) {
        const double d = in.dt[(int64_t)s * ld + t], sr = in.sog_rate[(int64_t)ui * ld + t],
                     cr = in.cog_rate ? in.cog_rate[(int64_t)ui * ld + t] : 0.0;
        status |= predict_core<NC>(a.p, Q, x, P, d, sr, cr, in.noise_pred ? in.noise_pred + (int64_t)s * n * ld + t : nullptr, ld,
                                   nullptr, nullptr, 0);
        if (in.upd_mask[(int64_t)s * ld + t]) {
            if (ui + 1 < a.max_obs) status |= update(++ui);
            else status |= STE_STATUS_OBS_OVERRUN;
        }
    }
    const int64_t row = (int64_t)c * a.scores.ld_out + t;
    a.scores.loglik[row] = loglik;
    a.scores.nis[row] = nis;
    a.scores.dof[row] = dof;
    a.scores.n_updates[row] = ui + 1;
    a.scores.status[row] = status;
}

// UnscentedKalmanFilter.rts_step (unscented.py:267-351) over ragged tracks: n_states = n_steps[t] + 1 and rate_repeat[t]
// per track; the status bits are OR-ed into the forward pass's.  Q as in the forward pass (PerTrack: noise.Q_tracks set).
template <int NC, bool PerTrack>
__global__ void __launch_bounds__(kThreadsN) urtss_backward_n_tracks_kernel(const __grid_constant__ FleetArgsN a) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= a.p.n_tracks) return;
    const SteInputsN &in = a.in;
    const int nt = in.n_steps ? min(in.n_steps[t], a.max_steps) : a.max_steps;
    const int rep = max(in.rate_repeat[t], 1);
    double Qt[PerTrack ? NC * NC : 1];
    const double *Q = track_matrix<NC, PerTrack>(a.p.Q, a.noise.Q_tracks, a.p.ld, t, Qt);
    a.out.status[t] |= rts_n<NC>(a.p, Q, t, nt + 1, rep, a.max_obs, a.out.mean_f, a.out.cov_f, in.dt, in.sog_rate, in.cog_rate,
                                 in.noise_bwd, a.out.mean_s, a.out.cov_s);
}

__global__ void __launch_bounds__(64) process_n_kernel(int model, int n, int T, int64_t ld, const double *xin, const double *dt,
                                                        const double *sog_rate, const double *cog_rate, double *xout) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    double x[kMaxN], y[kMaxN];
    for (int r = 0; r < n; ++r) x[r] = xin[r * ld + t];
    process_n(model, n, x, dt[t], sog_rate ? sog_rate[t] : 0.0, cog_rate ? cog_rate[t] : 0.0, y);
    for (int r = 0; r < n; ++r) xout[r * ld + t] = y[r];
}

// accuracy probe for ste_fastmath.cuh (tests only): out0/out1 = f(a, b)
__global__ void fastmath_probe_kernel(int kind, int n, const double *a, const double *b, double *out0, double *out1) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double r0 = 0.0, r1 = 0.0;
    switch (kind) {
        case 0: fast_sincos(a[i], &r0, &r1); break;
        case 1: r0 = fast_atan2<false>(a[i], b[i]); break;
        case 6: r0 = fast_atan2<true>(a[i], b[i]); break;
        case 2: r0 = fast_sqrt(a[i]); break;
        case 3: r0 = fast_rsqrt(a[i]); break;
        case 4: r0 = fast_rcp(a[i]); break;
        case 5: r0 = fast_div(a[i], b[i]); break;
        default: break;
    }
    out0[i] = r0;
    out1[i] = r1;
}

// FP64 pipe microbenchmark: CHAINS independent dependent chains per thread, clock64 timed.
// MODE 0: DFMA, register operands.  1: DFMA with a __constant__ (uniform-register) multiplicand.
// 2: DMUL + DADD alternating.  3: DFMA followed by a select on its result (DSETP + FSEL pair).
// 4: DFMA whose three source operands are three DIFFERENT registers that change every instruction
// (acc[k] = fma(acc[k], acc[k+1], acc[k+2])): what the filter's matrix code looks like to the register
// file, against mode 0 where two of the three operands never change.  5: the same with two sources (DMUL).
__constant__ double kProbeC[2] = {1.0000000001, 1e-12};
template <int CHAINS, int MODE>
__global__ void fp64_latency_probe_kernel(int iters, double *sink, long long *cycles) {
    double acc[CHAINS];
    const double a = 1.0 + 1e-9 * threadIdx.x, b = 1e-12;
#pragma unroll
    for (int k = 0; k < CHAINS; ++k) acc[k] = 0.1 * k;
    const long long t0 = clock64();
#pragma unroll 4
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < CHAINS; ++k) {
            if (MODE == 0) acc[k] = fma(acc[k], a, b);
            if (MODE == 1) acc[k] = fma(acc[k], kProbeC[0], kProbeC[1]);
            if (MODE == 2) acc[k] = (i & 1) ? acc[k] * a : acc[k] + b;
            if (MODE == 3) {
                const double v = fma(acc[k], a, b);
                acc[k] = (v > 1e300) ? b : v;
            }
            if (MODE == 4) acc[k] = fma(acc[k], acc[(k + 1) % CHAINS], -acc[(k + 2) % CHAINS]);
            if (MODE == 5) acc[k] = acc[k] * acc[(k + 1) % CHAINS];
        }
    }
    const long long t1 = clock64();
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < CHAINS; ++k) s += acc[k];
    sink[threadIdx.x] = s;
    if (threadIdx.x == 0) cycles[0] = t1 - t0;
}

__global__ void fp64_fma_probe_kernel(int iters, double *sink) {
    double acc[8];
    const double a = 1.0 + 1e-9 * threadIdx.x, b = 1e-12 * (blockIdx.x + 1);
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = 0.1 * k;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = fma(acc[k], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += acc[k];
    sink[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// ------------------------------------------------------------------------------------------ //
// host side of the ABI
// ------------------------------------------------------------------------------------------ //
static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, const char *detail = "") {
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}

static int check_launch(const char *what) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
        return STE_ERR_CUDA;
    }
    return STE_OK;
}

// the same two for the library's other translation units (ste_text.cu)
int report_error(int code, const char *what) { return fail(code, "%s", what); }
int report_launch(const char *what) { return check_launch(what); }

static bool is_symmetric(const double *M) {
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < i; ++j)
            if (M[i * 4 + j] != M[j * 4 + i]) return false;
    return true;
}

static bool is_symmetric_n(int n, const double *M) {
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j)
            if (M[i * n + j] != M[j * n + i]) return false;
    return true;
}

// H == diag(1,1,0,0) exactly and R zero outside its leading 2x2 block
static bool position_only(const SteProblem &p) {
    if (p.flags & STE_FLAG_FORCE_GENERIC) return false;
    for (int i = 0; i < 4; ++i)
        for (int j = 0; j < 4; ++j) {
            const double h = (i == j && i < 2) ? 1.0 : 0.0;
            if (p.H[i * 4 + j] != h) return false;
            if ((i >= 2 || j >= 2) && p.R[i * 4 + j] != 0.0) return false;
        }
    return true;
}

static int validate_problem(const SteProblem *p) {
    if (!p) return fail(STE_ERR_INVALID_ARG, "null SteProblem");
    if (p->n_tracks < 0 || p->max_steps < 0 || p->max_obs < 1) return fail(STE_ERR_INVALID_ARG, "negative sizes");
    if (p->ld < p->n_tracks) return fail(STE_ERR_INVALID_ARG, "ld < n_tracks");
    if (p->ld >= (1ll << 29)) return fail(STE_ERR_INVALID_ARG, "ld >= 2^29 (the kernels address planes with 32-bit byte strides)");
    if (!is_symmetric(p->Q) || !is_symmetric(p->R) || !is_symmetric(p->P0))
        return fail(STE_ERR_UNSUPPORTED, "Q, R and P0 must be symmetric");
    return STE_OK;
}

}  // namespace ste

using namespace ste;

extern "C" {

int ste_version(void) { return STE_ABI_VERSION; }

const char *ste_last_error(void) { return g_err; }

static int forward_input_rules(const SteProblem *prob, const SteInputs *in);

static int validate_forward(const SteProblem *prob, const SteInputs *in, const SteOutputs *out) {
    if (int rc = validate_problem(prob)) return rc;
    if (!in || !out) return fail(STE_ERR_INVALID_ARG, "null SteInputs/SteOutputs");
    if (!in->x0 || !in->dt || !in->sog_rate || !in->cog_rate) return fail(STE_ERR_INVALID_ARG, "missing input array");
    if (!out->mean_f || !out->cov_f || !out->status) return fail(STE_ERR_INVALID_ARG, "missing output array");
    return forward_input_rules(prob, in);
}

// what the forward pass requires of a tile's inputs beyond their presence: gating without measurement noise, the update
// variant a per-track R needs, and every observation row the update reads
static int forward_input_rules(const SteProblem *prob, const SteInputs *in) {
    const bool gating = (prob->flags & STE_FLAG_GATING) != 0;
    if (gating && in->noise_upd)
        return fail(STE_ERR_UNSUPPORTED, "gating draws a data-dependent number of normals; only zero measurement noise is supported with it");
    if (gating && prob->gate_max_iter < 1) return fail(STE_ERR_INVALID_ARG, "gate_max_iter < 1");
    const bool pos = position_only(*prob);
    if (in->R_tracks && pos)
        return fail(STE_ERR_INVALID_ARG, "a per-track R (SteInputs.R_tracks) needs the generic update: set STE_FLAG_FORCE_GENERIC");
    for (int r = 0; r < 4; ++r) {
        bool used = gating || in->R_tracks != nullptr;  // generic gating: y = z - x touches every row
        for (int j = 0; j < 4; ++j) used |= prob->H[r * 4 + j] != 0.0 || prob->R[r * 4 + j] != 0.0;
        if (pos) used = r < 2;  // rows 2, 3 only ever multiply exact zeros of pinv(S)
        if (used && !in->z[r]) return fail(STE_ERR_INVALID_ARG, "observation row referenced by H/R is NULL");
    }
    return STE_OK;
}

static int validate_backward(const SteProblem *prob, const SteInputs *in, const SteOutputs *out) {
    if (int rc = validate_problem(prob)) return rc;
    if (!in || !out) return fail(STE_ERR_INVALID_ARG, "null SteInputs/SteOutputs");
    if (!in->dt || !in->sog_rate || !in->cog_rate) return fail(STE_ERR_INVALID_ARG, "missing input array");
    if (!out->mean_f || !out->cov_f || !out->mean_s || !out->cov_s || !out->status)
        return fail(STE_ERR_INVALID_ARG, "missing output array");
    if ((out->mean_s == out->mean_f) != (out->cov_s == out->cov_f))
        return fail(STE_ERR_INVALID_ARG, "in-place smoothing must alias both mean and cov");
    return STE_OK;
}

static KernelArgs kernel_args(const SteProblem *prob, const SteInputs *in, const SteOutputs *out) {
    KernelArgs a;
    a.prob = *prob;
    a.in = *in;
    a.out = *out;
    return a;
}

static int validate_innovations(const SteInnovations *innov) {
    if (innov && (!innov->nis || !innov->loglik || !innov->rank))
        return fail(STE_ERR_INVALID_ARG, "SteInnovations needs all three planes (nis, loglik, rank)");
    return STE_OK;
}

extern "C++" {
template <bool POS_ONLY, bool GATING, bool INNOV, bool PER_Q>
static int launch_forward(const typename ForwardArgs<INNOV, PER_Q>::type &a, cudaStream_t s) {
    const dim3 grid((a.prob.n_tracks + kThreads - 1) / kThreads), block(kThreads);
    const size_t smem = sizeof(double) * kScratchSlotsFwd * kThreads;
    if (cudaFuncSetAttribute(ukf_forward_kernel<POS_ONLY, GATING, INNOV, PER_Q>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return check_launch("cudaFuncSetAttribute(ukf_forward_kernel)");
    ukf_forward_kernel<POS_ONLY, GATING, INNOV, PER_Q><<<grid, block, smem, s>>>(a);
    return check_launch("ukf_forward_kernel");
}

template <bool INNOV, bool PER_Q = false>
static int launch_forward(bool pos, bool gating, const typename ForwardArgs<INNOV, PER_Q>::type &a, cudaStream_t s) {
    if (pos) return gating ? launch_forward<true, true, INNOV, PER_Q>(a, s) : launch_forward<true, false, INNOV, PER_Q>(a, s);
    return gating ? launch_forward<false, true, INNOV, PER_Q>(a, s) : launch_forward<false, false, INNOV, PER_Q>(a, s);
}
}  // extern "C++"

int ste_ukf_forward_f64(const SteProblem *prob, const SteInputs *in, SteOutputs *out, void *stream) {
    return ste_ukf_forward_innov_f64(prob, in, nullptr, out, stream);
}

int ste_ukf_forward_innov_f64(const SteProblem *prob, const SteInputs *in, const SteInnovations *innov, SteOutputs *out,
                              void *stream) {
    if (int rc = validate_forward(prob, in, out)) return rc;
    if (int rc = validate_innovations(innov)) return rc;
    if (prob->n_tracks == 0) return STE_OK;
    const bool gating = (prob->flags & STE_FLAG_GATING) != 0, pos = position_only(*prob);
    cudaStream_t s = (cudaStream_t)stream;
    if (!innov) return launch_forward<false>(pos, gating, kernel_args(prob, in, out), s);
    KernelArgsInnov a;
    static_cast<KernelArgs &>(a) = kernel_args(prob, in, out);
    a.innov = *innov;
    return launch_forward<true>(pos, gating, a, s);
}

// the n = 4 passes' per-track noise: Q_tracks only (a per-track R travels in SteInputs.R_tracks)
static int validate_noise4(const SteNoiseN *noise) {
    if (noise && noise->R_tracks)
        return fail(STE_ERR_INVALID_ARG, "n = 4: a per-track R travels in SteInputs.R_tracks, not SteNoiseN.R_tracks");
    return STE_OK;
}

int ste_ukf_forward_noise_f64(const SteProblem *prob, const SteInputs *in, const SteNoiseN *noise, const SteInnovations *innov,
                              SteOutputs *out, void *stream) {
    if (int rc = validate_noise4(noise)) return rc;
    if (!noise || !noise->Q_tracks) return ste_ukf_forward_innov_f64(prob, in, innov, out, stream);
    if (int rc = validate_forward(prob, in, out)) return rc;
    if (int rc = validate_innovations(innov)) return rc;
    if (prob->n_tracks == 0) return STE_OK;
    const bool gating = (prob->flags & STE_FLAG_GATING) != 0, pos = position_only(*prob);
    KernelArgsQ a{};
    static_cast<KernelArgs &>(a) = kernel_args(prob, in, out);
    if (innov) a.innov = *innov;
    a.Q_tracks = noise->Q_tracks;
    cudaStream_t s = (cudaStream_t)stream;
    return innov ? launch_forward<true, true>(pos, gating, a, s) : launch_forward<false, true>(pos, gating, a, s);
}

// ------------------------------------------------------------------------------------------ //
// Noise-candidate scores (ste_ukf_score_f64 / ste_ukf_score_n_f64)
// ------------------------------------------------------------------------------------------ //
static int validate_candidates(const SteCandidates *cand, int n) {
    if (!cand || !cand->Q || !cand->R) return fail(STE_ERR_INVALID_ARG, "null SteCandidates table or matrix");
    if (cand->n_cand < 1 || cand->n_cand > STE_MAX_CANDIDATES)
        return fail(STE_ERR_INVALID_ARG, "SteCandidates.n_cand outside [1, STE_MAX_CANDIDATES]");
    for (int c = 0; c < cand->n_cand; ++c) {
        const double *Q = cand->Q + (size_t)c * n * n, *R = cand->R + (size_t)c * n * n;
        for (int k = 0; k < n * n; ++k)
            if (!std::isfinite(Q[k]) || !std::isfinite(R[k])) return fail(STE_ERR_UNSUPPORTED, "a candidate Q or R is not finite");
        if (!is_symmetric_n(n, Q) || !is_symmetric_n(n, R)) return fail(STE_ERR_UNSUPPORTED, "candidate Q and R must be symmetric");
    }
    return STE_OK;
}

static int validate_scores(const SteScores *sc, int32_t n_tracks) {
    if (!sc || !sc->loglik || !sc->nis || !sc->dof || !sc->n_updates || !sc->status)
        return fail(STE_ERR_INVALID_ARG, "SteScores needs all five planes (loglik, nis, dof, n_updates, status)");
    if (sc->ld_out < n_tracks) return fail(STE_ERR_INVALID_ARG, "SteScores.ld_out < n_tracks");
    return STE_OK;
}

extern "C++" {
template <bool POS_ONLY, bool GATING>
static int launch_score(const KernelArgsScore &a, int n_cand, cudaStream_t s) {
    const dim3 grid((a.prob.n_tracks + kThreads - 1) / kThreads, n_cand), block(kThreads);
    const size_t smem = sizeof(double) * kScratchSlotsFwd * kThreads;
    if (cudaFuncSetAttribute(ukf_score_kernel<POS_ONLY, GATING>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return check_launch("cudaFuncSetAttribute(ukf_score_kernel)");
    ukf_score_kernel<POS_ONLY, GATING><<<grid, block, smem, s>>>(a);
    return check_launch("ukf_score_kernel");
}
}  // extern "C++"

int ste_ukf_score_f64(const SteProblem *prob, const SteInputs *in, const SteCandidates *cand, SteScores *scores, void *stream) {
    if (!prob || !in) return fail(STE_ERR_INVALID_ARG, "null SteProblem / SteInputs");
    if (int rc = validate_candidates(cand, 4)) return rc;
    if (int rc = validate_scores(scores, prob->n_tracks)) return rc;
    if (in->R_tracks)
        return fail(STE_ERR_INVALID_ARG, "a tile with its own R (SteInputs.R_tracks) cannot be scored: the candidates replace R");
    KernelArgsScore a{};
    bool pos = false;
    for (int c = 0; c < cand->n_cand; ++c) {
        SteProblem pc = *prob;   // the tile as the forward pass would see it with candidate c
        memcpy(pc.Q, cand->Q + c * 16, sizeof(pc.Q));
        memcpy(pc.R, cand->R + c * 16, sizeof(pc.R));
        if (int rc = validate_problem(&pc)) return rc;
        if (!in->x0 || !in->dt || !in->sog_rate || !in->cog_rate) return fail(STE_ERR_INVALID_ARG, "missing input array");
        if (int rc = forward_input_rules(&pc, in)) return rc;
        const bool pc_pos = position_only(pc);
        if (c > 0 && pc_pos != pos)
            return fail(STE_ERR_UNSUPPORTED, "the candidates' R select different updates (position-only and generic): score them in separate calls");
        pos = pc_pos;
        memcpy(a.Q[c], pc.Q, sizeof(pc.Q));
        memcpy(a.R[c], pc.R, sizeof(pc.R));
    }
    if (prob->n_tracks == 0) return STE_OK;
    a.prob = *prob;
    a.in = *in;
    a.scores = *scores;
    const bool gating = (prob->flags & STE_FLAG_GATING) != 0;
    cudaStream_t s = (cudaStream_t)stream;
    if (pos) return gating ? launch_score<true, true>(a, cand->n_cand, s) : launch_score<true, false>(a, cand->n_cand, s);
    return gating ? launch_score<false, true>(a, cand->n_cand, s) : launch_score<false, false>(a, cand->n_cand, s);
}

extern "C++" {
template <bool PER_Q>
static int launch_backward(const typename ForwardArgs<false, PER_Q>::type &a, cudaStream_t s) {
    const dim3 grid((a.prob.n_tracks + kThreads - 1) / kThreads), block(kThreads);
    const size_t smem = sizeof(double) * kScratchSlotsBwd * kThreads;
    auto kernel = a.out.smooth_stats ? urtss_backward_kernel<true, PER_Q> : urtss_backward_kernel<false, PER_Q>;
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return check_launch("cudaFuncSetAttribute(urtss_backward_kernel)");
    kernel<<<grid, block, smem, s>>>(a);
    return check_launch("urtss_backward_kernel");
}
}  // extern "C++"

int ste_urtss_backward_f64(const SteProblem *prob, const SteInputs *in, SteOutputs *out, void *stream) {
    if (int rc = validate_backward(prob, in, out)) return rc;
    if (prob->n_tracks == 0) return STE_OK;
    return launch_backward<false>(kernel_args(prob, in, out), (cudaStream_t)stream);
}

int ste_urtss_backward_noise_f64(const SteProblem *prob, const SteInputs *in, const SteNoiseN *noise, SteOutputs *out,
                                 void *stream) {
    if (int rc = validate_noise4(noise)) return rc;
    if (!noise || !noise->Q_tracks) return ste_urtss_backward_f64(prob, in, out, stream);
    if (int rc = validate_backward(prob, in, out)) return rc;
    if (prob->n_tracks == 0) return STE_OK;
    KernelArgsQ a{};
    static_cast<KernelArgs &>(a) = kernel_args(prob, in, out);
    a.Q_tracks = noise->Q_tracks;
    return launch_backward<true>(a, (cudaStream_t)stream);
}

extern "C++" {
template <bool POS_ONLY, bool GATING>
static int launch_roles(const KernelArgs &a, const KernelArgs &b, cudaStream_t s) {
    RoleSplit split{(a.prob.n_tracks + kThreads - 1) / kThreads, (b.prob.n_tracks + kThreads - 1) / kThreads};
    const dim3 grid(split.blocks_a + split.blocks_b), block(kThreads);
    const size_t smem = sizeof(double) * kScratchSlots * kThreads;
    if (cudaFuncSetAttribute(ukf_roles_kernel<POS_ONLY, GATING>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return check_launch("cudaFuncSetAttribute(ukf_roles_kernel)");
    ukf_roles_kernel<POS_ONLY, GATING><<<grid, block, smem, s>>>(a, b, split);
    return check_launch("ukf_roles_kernel");
}
}  // extern "C++"

int ste_ukf_fused_f64(const SteProblem *fwd_prob, const SteInputs *fwd_in, SteOutputs *fwd_out,
                      const SteProblem *bwd_prob, const SteInputs *bwd_in, SteOutputs *bwd_out, void *stream) {
    if (int rc = validate_forward(fwd_prob, fwd_in, fwd_out)) return rc;
    if (int rc = validate_backward(bwd_prob, bwd_in, bwd_out)) return rc;
    if (fwd_out->mean_f == bwd_out->mean_f || fwd_out->mean_f == bwd_out->mean_s || fwd_out->status == bwd_out->status)
        return fail(STE_ERR_INVALID_ARG, "the two tiles of a fused pass must not share output arrays");
    if (fwd_prob->n_tracks == 0) return ste_urtss_backward_f64(bwd_prob, bwd_in, bwd_out, stream);
    if (bwd_prob->n_tracks == 0) return ste_ukf_forward_f64(fwd_prob, fwd_in, fwd_out, stream);
    const bool gating = (fwd_prob->flags & STE_FLAG_GATING) != 0, pos = position_only(*fwd_prob);
    const KernelArgs a = kernel_args(fwd_prob, fwd_in, fwd_out), b = kernel_args(bwd_prob, bwd_in, bwd_out);
    cudaStream_t s = (cudaStream_t)stream;
    if (pos) return gating ? launch_roles<true, true>(a, b, s) : launch_roles<true, false>(a, b, s);
    return gating ? launch_roles<false, true>(a, b, s) : launch_roles<false, false>(a, b, s);
}

int ste_ukf_predict_f64(const SteProblem *prob, double *x, double *P, const double *dt, const double *sog_rate,
                        const double *cog_rate, const double *noise, double *sigma_prior, double *sigma_post,
                        int32_t *status, void *stream) {
    if (int rc = validate_problem(prob)) return rc;
    if (!x || !P || !dt || !sog_rate || !cog_rate) return fail(STE_ERR_INVALID_ARG, "missing array");
    if ((sigma_prior == nullptr) != (sigma_post == nullptr))
        return fail(STE_ERR_INVALID_ARG, "sigma_prior and sigma_post must be given together");
    if (prob->n_tracks == 0) return STE_OK;
    StepArgs a{};
    a.prob = *prob;
    a.x = x; a.P = P; a.dt = dt; a.sog_rate = sog_rate; a.cog_rate = cog_rate; a.noise = noise;
    a.sigma_prior = sigma_prior; a.sigma_post = sigma_post; a.status = status;
    const dim3 grid((prob->n_tracks + kStepThreads - 1) / kStepThreads), block(kStepThreads);
    ukf_predict_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(a);
    return check_launch("ukf_predict_kernel");
}

int ste_ukf_update_f64(const SteProblem *prob, double *x, double *P, const double *z, const double *noise,
                       uint8_t *gate_iters, double *gate_lambda, double *gate_scale, int32_t *status, void *stream) {
    if (int rc = validate_problem(prob)) return rc;
    if (!x || !P || !z) return fail(STE_ERR_INVALID_ARG, "missing array");
    const bool gating = (prob->flags & STE_FLAG_GATING) != 0;
    if (gating && noise) return fail(STE_ERR_UNSUPPORTED, "gating supports zero measurement noise only");
    if (gating && prob->gate_max_iter < 1) return fail(STE_ERR_INVALID_ARG, "gate_max_iter < 1");
    if (prob->n_tracks == 0) return STE_OK;
    StepArgs a{};
    a.prob = *prob;
    a.x = x; a.P = P; a.z = z; a.noise = noise;
    a.gate_iters = gate_iters; a.gate_lambda = gate_lambda; a.gate_scale = gate_scale; a.status = status;
    const dim3 grid((prob->n_tracks + kThreads - 1) / kThreads), block(kThreads);
    cudaStream_t s = (cudaStream_t)stream;
    if (position_only(*prob)) {
        if (gating) ukf_update_kernel<true, true><<<grid, block, 0, s>>>(a);
        else ukf_update_kernel<true, false><<<grid, block, 0, s>>>(a);
    } else {
        if (gating) ukf_update_kernel<false, true><<<grid, block, 0, s>>>(a);
        else ukf_update_kernel<false, false><<<grid, block, 0, s>>>(a);
    }
    return check_launch("ukf_update_kernel");
}

static int model_dim_ok(int32_t n, int32_t model) {
    if (n < 1 || n > kMaxN) return fail(STE_ERR_UNSUPPORTED, "generic steps: 1 <= n <= 8");
    if (model == STE_MODEL_GEODETIC && n != 4) return fail(STE_ERR_UNSUPPORTED, "geodetic_dynamics has n = 4");
    if (model == STE_MODEL_GEODETIC_TURN && n != 5) return fail(STE_ERR_UNSUPPORTED, "geodetic_dynamics_turn has n = 5");
    if (model != STE_MODEL_GEODETIC && model != STE_MODEL_GEODETIC_TURN) return fail(STE_ERR_UNSUPPORTED, "unknown process model");
    return STE_OK;
}

int ste_ukf_predict_n_f64(int32_t n, int32_t model, int32_t n_tracks, int64_t ld, const double *Q_host, double *x, double *P,
                          const double *dt, const double *sog_rate, const double *cog_rate, const double *noise, double *sigma_prior,
                          double *sigma_post, int32_t *status, void *stream) {
    if (int rc = model_dim_ok(n, model)) return rc;
    if (n_tracks < 0 || ld < n_tracks) return fail(STE_ERR_INVALID_ARG, "bad n_tracks / ld");
    if (!Q_host || !x || !P || !dt) return fail(STE_ERR_INVALID_ARG, "missing array");
    if ((sigma_prior == nullptr) != (sigma_post == nullptr)) return fail(STE_ERR_INVALID_ARG, "sigma_prior and sigma_post must be given together");
    if (n_tracks == 0) return STE_OK;
    ProblemN p{};
    p.n = n; p.model = model; p.n_tracks = n_tracks; p.ld = ld;
    memcpy(p.Q, Q_host, sizeof(double) * n * n);
    ukf_predict_n_kernel<<<(n_tracks + 63) / 64, 64, 0, (cudaStream_t)stream>>>(p, x, P, dt, sog_rate, cog_rate, noise, sigma_prior, sigma_post, status);
    return check_launch("ukf_predict_n_kernel");
}

int ste_ukf_update_n_f64(int32_t n, int32_t n_tracks, int64_t ld, const double *H_host, const double *R_host, double *x, double *P,
                         const double *z, const double *noise, int32_t *status, void *stream) {
    if (n < 1 || n > kMaxN) return fail(STE_ERR_UNSUPPORTED, "generic steps: 1 <= n <= 8");
    if (n_tracks < 0 || ld < n_tracks) return fail(STE_ERR_INVALID_ARG, "bad n_tracks / ld");
    if (!H_host || !R_host || !x || !P || !z) return fail(STE_ERR_INVALID_ARG, "missing array");
    if (n_tracks == 0) return STE_OK;
    ProblemN p{};
    p.n = n; p.n_tracks = n_tracks; p.ld = ld;
    memcpy(p.H, H_host, sizeof(double) * n * n);
    memcpy(p.R, R_host, sizeof(double) * n * n);
    ukf_update_n_kernel<<<(n_tracks + 63) / 64, 64, 0, (cudaStream_t)stream>>>(p, x, P, z, noise, status);
    return check_launch("ukf_update_n_kernel");
}

int ste_urtss_backward_n_f64(int32_t n, int32_t model, int32_t n_tracks, int64_t ld, int32_t n_states, int32_t rate_repeat,
                             int32_t n_rates, const double *Q_host, const double *mean_f, const double *cov_f, const double *dt,
                             const double *sog_rate, const double *cog_rate, const double *noise, double *mean_s, double *cov_s,
                             int32_t *status, void *stream) {
    if (int rc = model_dim_ok(n, model)) return rc;
    if (n_tracks < 0 || ld < n_tracks) return fail(STE_ERR_INVALID_ARG, "bad n_tracks / ld");
    if (n_states < 1 || rate_repeat < 1 || n_rates < 1) return fail(STE_ERR_INVALID_ARG, "n_states, rate_repeat and n_rates must be >= 1");
    if (!Q_host || !mean_f || !cov_f || !mean_s || !cov_s || (n_states > 1 && !dt)) return fail(STE_ERR_INVALID_ARG, "missing array");
    if (mean_s == mean_f || cov_s == cov_f) return fail(STE_ERR_INVALID_ARG, "the generic smoother does not run in place");
    if (n_tracks == 0) return STE_OK;
    ProblemN p{};
    p.n = n; p.model = model; p.n_tracks = n_tracks; p.ld = ld;
    memcpy(p.Q, Q_host, sizeof(double) * n * n);
    urtss_backward_n_kernel<<<(n_tracks + 63) / 64, 64, 0, (cudaStream_t)stream>>>(p, n_states, rate_repeat, n_rates, mean_f, cov_f, dt,
                                                                                  sog_rate, cog_rate, noise, mean_s, cov_s, status);
    return check_launch("urtss_backward_n_kernel");
}

// the problem checks shared by the fleet passes and the five-state metrics
static int validate_problem_n(const SteProblemN *p) {
    if (p->model == STE_MODEL_GEODETIC && p->n == 4)
        return fail(STE_ERR_UNSUPPORTED, "n = 4 geodetic_dynamics runs on the batched n = 4 path: ste_ukf_forward_f64 / ste_urtss_backward_f64");
    if (int rc = model_dim_ok(p->n, p->model)) return rc;
    if (p->n != 5) return fail(STE_ERR_UNSUPPORTED, "the fleet kernels are built for n = 5 (geodetic_dynamics_turn)");
    if (p->n_tracks < 0 || p->max_steps < 0 || p->max_obs < 1) return fail(STE_ERR_INVALID_ARG, "negative sizes");
    if (p->ld < p->n_tracks) return fail(STE_ERR_INVALID_ARG, "ld < n_tracks");
    if (!is_symmetric_n(p->n, p->Q) || !is_symmetric_n(p->n, p->R) || !is_symmetric_n(p->n, p->P0))
        return fail(STE_ERR_UNSUPPORTED, "Q, R and P0 must be symmetric");
    return STE_OK;
}

static int validate_fleet_n(const SteProblemN *p, const SteInputsN *in, const SteOutputsN *out, bool backward) {
    if (!p || !in || !out) return fail(STE_ERR_INVALID_ARG, "null SteProblemN / SteInputsN / SteOutputsN");
    if (int rc = validate_problem_n(p)) return rc;
    if (!in->dt || !in->sog_rate || (!backward && (!in->x0 || !in->upd_mask)) || (backward && !in->rate_repeat))
        return fail(STE_ERR_INVALID_ARG, "missing input array");
    if (!out->mean_f || !out->cov_f || !out->status || (backward && (!out->mean_s || !out->cov_s)))
        return fail(STE_ERR_INVALID_ARG, "missing output array");
    if ((out->mean_s && (out->mean_s == out->mean_f || out->mean_s == out->cov_f)) ||
        (out->cov_s && (out->cov_s == out->cov_f || out->cov_s == out->mean_f)))
        return fail(STE_ERR_INVALID_ARG, "mean_s / cov_s must not alias the filtered arrays");
    return STE_OK;
}

static FleetArgsN fleet_args(const SteProblemN *prob, const SteInputsN *in, const SteOutputsN *out, const SteNoiseN *noise) {
    FleetArgsN a{};
    const int n = prob->n;
    a.p.n = n; a.p.model = prob->model; a.p.n_tracks = prob->n_tracks; a.p.ld = prob->ld;
    memcpy(a.p.H, prob->H, sizeof(double) * n * n);
    memcpy(a.p.Q, prob->Q, sizeof(double) * n * n);
    memcpy(a.p.R, prob->R, sizeof(double) * n * n);
    memcpy(a.P0, prob->P0, sizeof(double) * n * n);
    a.max_steps = prob->max_steps; a.max_obs = prob->max_obs;
    a.in = *in;
    a.out = *out;
    if (noise) a.noise = *noise;
    return a;
}

int ste_ukf_forward_n_f64(const SteProblemN *prob, const SteInputsN *in, SteOutputsN *out, void *stream) {
    return ste_ukf_forward_noise_n_f64(prob, in, nullptr, out, stream);
}

int ste_ukf_forward_noise_n_f64(const SteProblemN *prob, const SteInputsN *in, const SteNoiseN *noise, SteOutputsN *out,
                                void *stream) {
    return ste_ukf_forward_innov_n_f64(prob, in, noise, nullptr, out, stream);
}

int ste_ukf_forward_innov_n_f64(const SteProblemN *prob, const SteInputsN *in, const SteNoiseN *noise,
                                const SteInnovations *innov, SteOutputsN *out, void *stream) {
    if (int rc = validate_fleet_n(prob, in, out, false)) return rc;
    if (int rc = validate_innovations(innov)) return rc;
    if (prob->n_tracks == 0) return STE_OK;
    FleetArgsN a = fleet_args(prob, in, out, noise);
    const int blocks = (prob->n_tracks + kThreadsN - 1) / kThreadsN;
    cudaStream_t s = (cudaStream_t)stream;
    const bool per_track = a.noise.Q_tracks || a.noise.R_tracks;
    if (innov) {
        a.innov = *innov;
        if (per_track) ukf_forward_n_kernel<5, true, true><<<blocks, kThreadsN, 0, s>>>(a);
        else ukf_forward_n_kernel<5, false, true><<<blocks, kThreadsN, 0, s>>>(a);
    } else if (per_track) {
        ukf_forward_n_kernel<5, true><<<blocks, kThreadsN, 0, s>>>(a);
    } else {
        ukf_forward_n_kernel<5, false><<<blocks, kThreadsN, 0, s>>>(a);
    }
    return check_launch("ukf_forward_n_kernel");
}

int ste_ukf_score_n_f64(const SteProblemN *prob, const SteInputsN *in, const SteCandidates *cand, SteScores *scores, void *stream) {
    if (!prob || !in) return fail(STE_ERR_INVALID_ARG, "null SteProblemN / SteInputsN");
    if (int rc = validate_candidates(cand, 5)) return rc;
    if (int rc = validate_scores(scores, prob->n_tracks)) return rc;
    ScoreArgsN a{};
    for (int c = 0; c < cand->n_cand; ++c) {
        SteProblemN pc = *prob;   // the tile as the forward pass would see it with candidate c
        memcpy(pc.Q, cand->Q + c * 25, sizeof(double) * 25);
        memcpy(pc.R, cand->R + c * 25, sizeof(double) * 25);
        if (int rc = validate_problem_n(&pc)) return rc;
        memcpy(a.Q[c], pc.Q, sizeof(a.Q[c]));
        memcpy(a.R[c], pc.R, sizeof(a.R[c]));
    }
    if (!in->x0 || !in->dt || !in->sog_rate || !in->upd_mask) return fail(STE_ERR_INVALID_ARG, "missing input array");
    if (prob->n_tracks == 0) return STE_OK;
    const int n = prob->n;
    a.p.n = n; a.p.model = prob->model; a.p.n_tracks = prob->n_tracks; a.p.ld = prob->ld;
    memcpy(a.p.H, prob->H, sizeof(double) * n * n);
    memcpy(a.p.Q, prob->Q, sizeof(double) * n * n);
    memcpy(a.p.R, prob->R, sizeof(double) * n * n);
    memcpy(a.P0, prob->P0, sizeof(double) * n * n);
    a.max_steps = prob->max_steps; a.max_obs = prob->max_obs;
    a.in = *in;
    a.scores = *scores;
    const dim3 grid((prob->n_tracks + kThreadsN - 1) / kThreadsN, cand->n_cand);
    ukf_score_n_kernel<5><<<grid, kThreadsN, 0, (cudaStream_t)stream>>>(a);
    return check_launch("ukf_score_n_kernel");
}

int ste_urtss_backward_tracks_n_f64(const SteProblemN *prob, const SteInputsN *in, SteOutputsN *out, void *stream) {
    return ste_urtss_backward_tracks_noise_n_f64(prob, in, nullptr, out, stream);
}

int ste_urtss_backward_tracks_noise_n_f64(const SteProblemN *prob, const SteInputsN *in, const SteNoiseN *noise,
                                          SteOutputsN *out, void *stream) {
    if (int rc = validate_fleet_n(prob, in, out, true)) return rc;
    if (prob->n_tracks == 0) return STE_OK;
    const FleetArgsN a = fleet_args(prob, in, out, noise);
    const int blocks = (prob->n_tracks + kThreadsN - 1) / kThreadsN;
    if (a.noise.Q_tracks)
        urtss_backward_n_tracks_kernel<5, true><<<blocks, kThreadsN, 0, (cudaStream_t)stream>>>(a);
    else
        urtss_backward_n_tracks_kernel<5, false><<<blocks, kThreadsN, 0, (cudaStream_t)stream>>>(a);
    return check_launch("urtss_backward_n_tracks_kernel");
}

int ste_process_f64(int32_t model, int32_t n, int32_t n_tracks, int64_t ld, const double *x_in, const double *dt,
                    const double *sog_rate, const double *cog_rate, double *x_out, void *stream) {
    if (int rc = model_dim_ok(n, model)) return rc;
    if (n_tracks < 0 || ld < n_tracks) return fail(STE_ERR_INVALID_ARG, "bad n_tracks / ld");
    if (!x_in || !dt || !x_out) return fail(STE_ERR_INVALID_ARG, "missing array");
    if (n_tracks == 0) return STE_OK;
    process_n_kernel<<<(n_tracks + 63) / 64, 64, 0, (cudaStream_t)stream>>>(model, n, n_tracks, ld, x_in, dt, sog_rate, cog_rate, x_out);
    return check_launch("process_n_kernel");
}

int ste_csv_parse_rows(const uint8_t *bytes, const int64_t *row_start, int64_t n_rows, const int32_t *cols_host, int64_t *hours,
                       double *lat, double *lon, uint64_t *id_key, int64_t *id_int, int32_t *id_off, int32_t *id_len, int64_t *label,
                       int32_t *flags, void *stream) {
    if (n_rows < 0) return fail(STE_ERR_INVALID_ARG, "negative row count");
    if (!bytes || !row_start || !cols_host || !hours || !lat || !lon || !id_key || !id_int || !id_off || !id_len || !label || !flags)
        return fail(STE_ERR_INVALID_ARG, "missing array");
    for (int k = 0; k < kCsvColLabel; ++k)
        if (cols_host[k] < 0) return fail(STE_ERR_INVALID_ARG, "yr, mo, dy, hr, lat, lon and id columns are required");
    if (n_rows == 0) return STE_OK;
    CsvArgs a{};
    a.bytes = bytes; a.row_start = row_start; a.n_rows = n_rows;
    for (int k = 0; k < kCsvTargets; ++k) a.cols[k] = cols_host[k];
    a.hours = hours; a.lat = lat; a.lon = lon; a.id_key = id_key; a.id_int = id_int; a.id_off = id_off; a.id_len = id_len;
    a.label = label; a.flags = flags;
    const int64_t blocks = (n_rows + 255) / 256;
    if (blocks > 0x7fffffffll) return fail(STE_ERR_UNSUPPORTED, "more than 2^31 blocks of rows: split the file");
    csv_parse_rows_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a);
    return check_launch("csv_parse_rows_kernel");
}

int ste_gate_terms_f64(const SteProblem *prob, const double *x, const double *P, const double *z, double *gamma, double *denom,
                       void *stream) {
    if (int rc = validate_problem(prob)) return rc;
    if (!x || !P || !z || !gamma || !denom) return fail(STE_ERR_INVALID_ARG, "missing array");
    if (prob->n_tracks == 0) return STE_OK;
    StepArgs a{};
    a.prob = *prob;
    a.x = const_cast<double *>(x); a.P = const_cast<double *>(P); a.z = z;
    const dim3 grid((prob->n_tracks + kThreads - 1) / kThreads), block(kThreads);
    gate_terms_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(a, gamma, denom);
    return check_launch("gate_terms_kernel");
}

int ste_sigma_points_f64(int32_t n, int32_t n_tracks, int64_t ld, double scale, const double *x, const double *P,
                         double *X, int32_t *status, void *stream) {
    if (n < 1 || n > 8) return fail(STE_ERR_UNSUPPORTED, "sigma points: 1 <= n <= 8");
    if (n_tracks < 0 || ld < n_tracks) return fail(STE_ERR_INVALID_ARG, "bad n_tracks / ld");
    if (!x || !P || !X) return fail(STE_ERR_INVALID_ARG, "missing array");
    if (n_tracks == 0) return STE_OK;
    const dim3 grid((n_tracks + kThreads - 1) / kThreads), block(kThreads);
    sigma_points_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(n, n_tracks, ld, scale, x, P, X, status);
    return check_launch("sigma_points_kernel");
}

int ste_geodetic_f64(int32_t n_tracks, int64_t ld, const double *x_in, const double *dt, const double *sog_rate,
                     const double *cog_rate, double *x_out, void *stream) {
    if (n_tracks < 0 || ld < n_tracks) return fail(STE_ERR_INVALID_ARG, "bad n_tracks / ld");
    if (!x_in || !dt || !sog_rate || !cog_rate || !x_out) return fail(STE_ERR_INVALID_ARG, "missing array");
    if (n_tracks == 0) return STE_OK;
    const dim3 grid((n_tracks + kThreads - 1) / kThreads), block(kThreads);
    geodetic_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(n_tracks, ld, x_in, dt, sog_rate, cog_rate, x_out);
    return check_launch("geodetic_kernel");
}

int ste_derive_inputs_f64(int32_t n_tracks, int32_t max_obs, int64_t ld, int32_t smooth_width, int32_t geodesy, const double *lon,
                          const double *lat, const double *dts, const int32_t *n_obs, double *sog, double *cog,
                          double *sog_rate, double *cog_rate, void *stream) {
    if (n_tracks < 0 || max_obs < 2 || ld < n_tracks) return fail(STE_ERR_INVALID_ARG, "bad n_tracks / max_obs / ld");
    if (smooth_width < 0 || smooth_width > 64) return fail(STE_ERR_INVALID_ARG, "smooth_width outside [0, 64]");
    if (geodesy != STE_GEODESY_SPHERE && geodesy != STE_GEODESY_WGS84) return fail(STE_ERR_INVALID_ARG, "unknown geodesy");
    if (!lon || !lat || !dts || !sog || !cog || !sog_rate || !cog_rate) return fail(STE_ERR_INVALID_ARG, "missing array");
    if (n_tracks == 0) return STE_OK;
    const dim3 grid((n_tracks + kThreads - 1) / kThreads), block(kThreads);
    derive_inputs_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(n_tracks, max_obs, ld, smooth_width, geodesy, lon, lat, dts, n_obs, sog,
                                                                  cog, sog_rate, cog_rate);
    return check_launch("derive_inputs_kernel");
}

extern "C++" {
template <int NS>
static int launch_track_metrics(const MetricsArgs<NS> &a, cudaStream_t s) {
    int rows = 0;
    for (int r = 0; r < NS; ++r) rows += a.in.z[r] != nullptr;
    if (rows == 0) return fail(STE_ERR_INVALID_ARG, "no observation row to compare with");
    const dim3 grid((a.prob.n_tracks + kThreads - 1) / kThreads, rows), block(kThreads);
    track_metrics_kernel<NS><<<grid, block, 0, s>>>(a);
    return check_launch("track_metrics_kernel");
}
}

int ste_track_metrics_f64(const SteProblem *prob, const SteInputs *in, const double *mean, double *rmse, double *cum_abs,
                          double *max_abs, double *abs_diff, int32_t *n_pairs, void *stream) {
    if (int rc = validate_problem(prob)) return rc;
    if (!in || !mean) return fail(STE_ERR_INVALID_ARG, "null SteInputs / state array");
    if (prob->n_tracks == 0) return STE_OK;
    MetricsArgs<4> a{};
    a.prob = *prob;
    a.in = *in;
    a.mean = mean; a.rmse = rmse; a.cum_abs = cum_abs; a.max_abs = max_abs; a.abs_diff = abs_diff; a.n_pairs = n_pairs;
    return launch_track_metrics(a, (cudaStream_t)stream);
}

int ste_track_metrics_n_f64(const SteProblemN *prob, const SteInputsN *in, const double *mean, double *rmse, double *cum_abs,
                            double *max_abs, double *abs_diff, int32_t *n_pairs, void *stream) {
    if (!prob || !in) return fail(STE_ERR_INVALID_ARG, "null SteProblemN / SteInputsN");
    if (int rc = validate_problem_n(prob)) return rc;
    if (!in->upd_mask) return fail(STE_ERR_INVALID_ARG, "missing input array");
    if (!mean) return fail(STE_ERR_INVALID_ARG, "null state array");
    if (prob->n_tracks == 0) return STE_OK;
    MetricsArgs<5> a{};
    a.prob = *prob;
    a.in = *in;
    a.mean = mean; a.rmse = rmse; a.cum_abs = cum_abs; a.max_abs = max_abs; a.abs_diff = abs_diff; a.n_pairs = n_pairs;
    return launch_track_metrics(a, (cudaStream_t)stream);
}

int ste_probe_fastmath(int32_t kind, int32_t n, const double *a, const double *b, double *out0, double *out1, void *stream) {
    if (kind < 0 || kind > 6 || n < 0 || !a || !b || !out0 || !out1) return fail(STE_ERR_INVALID_ARG, "bad fastmath probe arguments");
    if (n == 0) return STE_OK;
    fastmath_probe_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(kind, n, a, b, out0, out1);
    return check_launch("fastmath_probe_kernel");
}

int ste_probe_fp64_latency(int32_t warps, int32_t iters, int32_t chains, double *sink, long long *cycles, void *stream) {
    if (warps < 1 || warps > 32 || iters < 1 || chains < 1 || !sink || !cycles)
        return fail(STE_ERR_INVALID_ARG, "bad latency probe arguments");
    cudaStream_t s = (cudaStream_t)stream;
    const int mode = chains / 100;   // chains = 100 * mode + {1, 2, 4, 8}
    const int ch = chains % 100;
#define STE_PROBE_CASE(C_, M_) if (ch == C_ && mode == M_) { fp64_latency_probe_kernel<C_, M_><<<1, 32 * warps, 0, s>>>(iters, sink, cycles); return check_launch("fp64_latency_probe_kernel"); }
    STE_PROBE_CASE(1, 0) STE_PROBE_CASE(2, 0) STE_PROBE_CASE(4, 0) STE_PROBE_CASE(8, 0)
    STE_PROBE_CASE(1, 1) STE_PROBE_CASE(4, 1) STE_PROBE_CASE(8, 1)
    STE_PROBE_CASE(1, 2) STE_PROBE_CASE(4, 2) STE_PROBE_CASE(8, 2)
    STE_PROBE_CASE(1, 3) STE_PROBE_CASE(4, 3) STE_PROBE_CASE(8, 3)
    STE_PROBE_CASE(4, 4) STE_PROBE_CASE(8, 4) STE_PROBE_CASE(4, 5) STE_PROBE_CASE(8, 5)
#undef STE_PROBE_CASE
    return fail(STE_ERR_INVALID_ARG, "chains must be 100 * mode + {1, 2, 4, 8}");
    return check_launch("fp64_latency_probe_kernel");
}

int ste_probe_fp64_fma(int32_t blocks, int32_t threads, int32_t iters, double *sink, void *stream) {
    if (blocks < 1 || threads < 1 || threads > 1024 || iters < 1 || !sink)
        return fail(STE_ERR_INVALID_ARG, "bad probe arguments");
    fp64_fma_probe_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(iters, sink);
    return check_launch("fp64_fma_probe_kernel");
}

}  // extern "C"
