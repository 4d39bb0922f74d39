/*
 * ste_ukf.h - C ABI of the B200-native batched UKF + URTSS library (libste_ukf.so).
 *
 * The reference (NOC-OI/ship-track-estimators) is pure Python and has no FFI layer; the
 * "operator interface" this ABI sits behind is the Python class API of
 *   src/track_estimators/kalman_filters/unscented.py   (UnscentedKalmanFilter)
 *   src/track_estimators/kalman_filters/kalman_filter.py (KalmanFilterBase.run / run_rts_smoother)
 *   src/track_estimators/kalman_filters/non_linear_process.py (geodetic_dynamics)
 * Each entry point names the reference function(s) it replaces.  A maintainer binds it with
 * ctypes (see INTEGRATION.md); the shipped binding is ship_track_estimators_b200/_native.py.
 *
 * Conventions
 *  - n = 4 state [lon deg, lat deg, SOG km/h, COG deg]; time in hours; all arithmetic fp64.
 *  - Every array is structure-of-arrays with the TRACK index fastest: element (plane, t) lives at
 *    base[plane * ld + t], ld >= n_tracks ("leading dimension", lets a launch address a
 *    sub-range of a larger allocation).  Matrices are row-major planes: P[i][j] is plane i*4+j.
 *  - Pointers are DEVICE pointers unless stated; the caller (torch) owns every buffer.  The
 *    library allocates nothing persistent and never frees caller memory.
 *  - Calls are asynchronous on the given CUDA stream (a cudaStream_t passed as void*; NULL =
 *    legacy default stream) and never synchronise.  Stateless and re-entrant.
 *  - Return value: 0 = launched; negative = STE_ERR_* (nothing launched).  Per-track numerical
 *    events go to the status[] output, never to the return code.  ste_last_error() returns a
 *    thread-local message for the last non-zero return.
 *  - There is no CPU fallback anywhere behind this ABI.
 */
#ifndef STE_UKF_H
#define STE_UKF_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STE_ABI_VERSION 7   /* 2: ste_ukf_fused_f64, ste_track_metrics_f64, geodesy argument of ste_derive_inputs_f64, STE_FLAG_LONG_STEPS */
                            /* 3: smooth_stats holds STE_STATS_PLANES = 15 planes per step (was 30)                                          */
                            /* 4: SteInputs.R_tracks, dimension-generic steps (ste_ukf_*_n_f64, ste_process_f64), ste_gate_terms_f64          */
                            /* 5: ste_urtss_backward_n_f64 (dimension-generic smoother); ld < 2^29                                            */
                            /* 6: fleet path of the five-state model: SteProblemN / SteInputsN / SteOutputsN, ste_ukf_forward_n_f64,      */
                            /*    ste_urtss_backward_tracks_n_f64                                                                          */
                            /* 7: ste_track_metrics_n_f64 (fit metrics of the five-state fleet path)                                      */
                            /*    additive, no struct changed: SteNoiseN, ste_ukf_forward_noise_n_f64,                                    */
                            /*    ste_urtss_backward_tracks_noise_n_f64 (per-track Q / R of the five-state fleet path)                    */
#define STE_STATS_PLANES 15
#define STE_DIM 4
#define STE_NSIGMA 9

/* return codes */
#define STE_OK 0
#define STE_ERR_INVALID_ARG (-1)
#define STE_ERR_CUDA (-2)
#define STE_ERR_UNSUPPORTED (-3)

/* SteProblem.flags */
#define STE_FLAG_GATING 0x1u      /* Mahalanobis robustification before every update            */
#define STE_FLAG_FORCE_GENERIC 0x2u /* never take the position-only (H = diag(1,1,0,0)) fast path */
#define STE_FLAG_PACKED_COV 0x4u  /* cov_f / cov_s hold the 10 unique entries per state, planes in  */
                                  /* the order 00 01 02 03 11 12 13 22 23 33, instead of 16         */
#define STE_FLAG_LONG_STEPS 0x8u  /* never take the small-displacement tier of the geodetic step     */
                                  /* (<= 100 km per predict below 75 deg latitude, decided per step  */
                                  /* and track): for tiles mixing short and long steps, where the    */
                                  /* lanes of a warp would otherwise split between the two tiers     */

/* per-track status bits (SteOutputs.status) */
#define STE_STATUS_NONFINITE 0x1     /* a state or covariance entry became NaN/Inf                  */
#define STE_STATUS_INDEFINITE 0x2    /* a covariance had a negative eigenvalue at a square root;    */
                                     /* the reference keeps Re(sqrtm) = root of the clamped spectrum */
#define STE_STATUS_GATE_CAP 0x4      /* robustification hit gate_max_iter                           */
#define STE_STATUS_OBS_OVERRUN 0x8   /* more update times matched than observations exist           */
                                     /* (the reference raises IndexError; the host binding does too) */
#define STE_STATUS_RANK_DEFICIENT 0x10 /* a pseudo-inverse dropped a non-structural singular value  */
#define STE_STATUS_SMOOTH_RECOMPUTE 0x100 /* informational: the step grid of this track does not let  */
                                     /* the smoother reuse the filter's statistics; it recomputes   */

/*
 * Problem description shared by all tracks of a launch ("tile").
 * H, Q, R, P0: reference UnscentedKalmanFilter.__init__ (unscented.py:20-74).  Q, R, P0 must be
 * symmetric.
 */
typedef struct SteProblem {
    int32_t n_tracks;      /* T                                                             */
    int32_t max_steps;     /* N_max: filter steps of the longest track (states = N_max + 1) */
    int32_t max_obs;       /* rows available in the observation arrays                      */
    int32_t substeps;      /* k >= 1: used when upd_mask == NULL: step s assimilates an     */
                           /* observation iff (s + 1) % k == 0                              */
    int32_t rate_repeat;   /* backward pass reads rate[step / rate_repeat] when the         */
                           /* per-track array is NULL (unscented.py:287-292)                */
    uint32_t flags;        /* STE_FLAG_*                                                    */
    int32_t gate_max_iter; /* cap on robustification iterations (reference: unbounded)      */
    int32_t reserved;      /* must be 0                                                     */
    int64_t ld;            /* leading dimension of every SoA array (>= n_tracks, < 2^29)    */
    double gate_chi;       /* chi_alpha, reference value 50 (unscented.py:357)              */
    double H[16];
    double Q[16];
    double R[16];
    double P0[16];
} SteProblem;

/* Inputs of the forward and backward passes (reference: the ShipTrack attributes read at
 * kalman_filter.py:73-108 and unscented.py:287-311, plus the dt array of run()). */
typedef struct SteInputs {
    const double *x0;        /* [4][ld] initial state (reference: x0 = z[:, 0])                   */
    const double *P0;        /* [16][ld] per-track prior covariance, or NULL -> SteProblem.P0    */
    const double *dt;        /* [max_steps][ld] step lengths (hours)                              */
    const uint8_t *upd_mask; /* [max_steps][ld] 1 = step ends exactly on an observation time      */
                             /* (kalman_filter.py:101), or NULL -> SteProblem.substeps cadence   */
    const int32_t *n_steps;  /* [T] steps per track, or NULL -> max_steps for all                */
    const double *z[4];      /* [max_obs][ld] observation rows lon, lat, sog, cog.  A row may be */
                             /* NULL when neither H nor R reference it (it is then read as 0)   */
    const double *sog_rate;  /* [max_obs][ld]                                                     */
    const double *cog_rate;  /* [max_obs][ld]                                                     */
    const int32_t *rate_repeat; /* [T] backward-pass rate repeat per track, or NULL             */
    /* optional noise tapes of UNIT normals (NULL = zero noise), scaled on the device by        */
    /* sqrt(diag Q) / sqrt(diag R) as np.random.normal(scale=...) does                           */
    const double *noise_pred; /* [max_steps][4][ld]  unscented.py:198-202                        */
    const double *noise_upd;  /* [max_obs][4][ld]    unscented.py:232-236, row = update index    */
    const double *noise_bwd;  /* [max_steps][4][ld]  unscented.py:320-323, row = backward step   */
    const double *R_tracks;   /* [16][ld] per-track measurement covariance (row-major 4x4 planes,  */
                              /* symmetric), or NULL -> SteProblem.R for every track.  Needs the   */
                              /* generic update: set STE_FLAG_FORCE_GENERIC (ABI 4)                */
} SteInputs;

typedef struct SteOutputs {
    double *mean_f;      /* [max_steps+1][4][ld]  filtered means; row 0 = prior (kalman_filter.py:76) */
    double *cov_f;       /* [max_steps+1][16][ld] filtered covariances ([..][10][ld] if PACKED_COV)   */
    double *mean_s;      /* smoothed, same shapes (may alias mean_f / cov_f for in-place smoothing)  */
    double *cov_s;
    int32_t *status;     /* [T] OR-ed STE_STATUS_* (the forward pass overwrites, the backward ORs)    */
    int32_t *n_updates;  /* [T] observations assimilated incl. the initial one, or NULL               */
    uint8_t *gate_iters; /* [max_obs][ld] robustification iterations per update, or NULL              */
    double *gate_lambda; /* [max_obs][ld] final lambda factor per update, or NULL                     */
    double *gate_scale;  /* [max_obs][ld] accumulated scale of R (product of lambdas), or NULL        */
    double *smooth_stats; /* [max_steps][STE_STATS_PLANES][ld] or NULL.  Written by the forward pass,  */
                         /* read by the backward pass: per predict step the noise-free predicted-mean */
                         /* offset (4), the predicted covariance about the filtered mean (3 entries)  */
                         /* and the cross covariance (8 entries) that rts_step recomputes from the    */
                         /* same sigma points (unscented.py:299-330); the entries that follow from    */
                         /* the filtered covariance (linear speed / course rows) are not stored.      */
                         /* NULL: the backward pass recomputes them.                                  */
} SteOutputs;

/* library / device -------------------------------------------------------------------------- */
int ste_version(void);
const char *ste_last_error(void);

/* KalmanFilterBase.run (kalman_filter.py:36-117) with UnscentedKalmanFilter.predict / update
 * (unscented.py:144-265) [+ check_robustness :353-511 when STE_FLAG_GATING] for T tracks. */
int ste_ukf_forward_f64(const SteProblem *prob, const SteInputs *in, SteOutputs *out, void *stream);

/* UnscentedKalmanFilter.rts_step (unscented.py:267-351) for T tracks; reads mean_f/cov_f
 * written by the forward pass, writes mean_s/cov_s. */
int ste_urtss_backward_f64(const SteProblem *prob, const SteInputs *in, SteOutputs *out, void *stream);

/* The loop of examples/example_ukf_rts_smoother_batch.py:19-71 over successive tiles of tracks,
 * software-pipelined: ONE launch runs KalmanFilterBase.run for the tracks of tile `fwd_*` and
 * UnscentedKalmanFilter.rts_step (all steps) for the tracks of tile `bwd_*`, which an earlier
 * call has already filtered (forward pass or fused pass).  The blocks of the launch take the
 * filter's or the smoother's role, interleaved so that every SM holds both.  Results are
 * bit-identical to ste_ukf_forward_f64(fwd) followed by ste_urtss_backward_f64(bwd).  Measured
 * on B200 it is ~13 % slower than those two launches back to back (two instruction streams per
 * SM overflow the instruction cache, DESIGN.md section 4): an entry point for callers that want
 * one launch per tile, not the fast path.  The two tiles must use different output arrays;
 * either may be empty (n_tracks == 0). */
int ste_ukf_fused_f64(const SteProblem *fwd_prob, const SteInputs *fwd_in, SteOutputs *fwd_out,
                      const SteProblem *bwd_prob, const SteInputs *bwd_in, SteOutputs *bwd_out, void *stream);

/* One UnscentedKalmanFilter.predict (unscented.py:144-207) for T independent filters, in place.
 * x [4][ld], P [16][ld], dt/sog_rate/cog_rate [T]; noise [4][ld] unit normals or NULL;
 * sigma_prior / sigma_post [36][ld] (plane = row*9 + point) or NULL; status [T] or NULL. */
int ste_ukf_predict_f64(const SteProblem *prob, double *x, double *P, const double *dt,
                        const double *sog_rate, const double *cog_rate, const double *noise,
                        double *sigma_prior, double *sigma_post, int32_t *status, void *stream);

/* One UnscentedKalmanFilter.update (unscented.py:209-265) for T filters, in place.
 * z [4][ld]; noise [4][ld] or NULL; gate_iters / gate_lambda / gate_scale [T] or NULL
 * (check_robustness, unscented.py:353-387: R_scaled = R * gate_scale). */
int ste_ukf_update_f64(const SteProblem *prob, double *x, double *P, const double *z,
                       const double *noise, uint8_t *gate_iters, double *gate_lambda,
                       double *gate_scale, int32_t *status, void *stream);

/* Dimension-generic single steps: the reference's class takes n from H (unscented.py:52-62) and any process
 * callable; these entry points serve that surface for n <= 8 and the process models the library ships.
 *   STE_MODEL_GEODETIC        n = 4  geodetic_dynamics, rates from the sog_rate / cog_rate arguments
 *   STE_MODEL_GEODETIC_TURN   n = 5  [lon, lat, sog, cog, cog_rate]: the geodetic step with the turn rate taken from
 *                                    the state, where it persists (the cog_rate argument is ignored, may be NULL)
 * (the reference's default weight W0 = 1 - n/3 must lie in (-1, 1), unscented.py:125-129: its class runs n <= 5)
 * H, Q, R are HOST pointers to row-major n x n matrices (they travel in the kernel parameters).
 * ste_ukf_predict_n_f64: UnscentedKalmanFilter.predict (unscented.py:144-207): x [n][ld], P [n*n][ld] in place;
 *   dt [T]; noise [n][ld] unit normals or NULL; sigma_prior / sigma_post [n*(2n+1)][ld] or NULL; status [T] or NULL.
 * ste_ukf_update_n_f64: UnscentedKalmanFilter.update (unscented.py:209-265) with dense H and R; state index 3 is
 *   the heading (innovation wrapped to [-180, 180), state taken modulo 360) as the reference hard-codes (:250, 257).
 * ste_urtss_backward_n_f64: UnscentedKalmanFilter.rts_step (unscented.py:267-351), the whole backward loop of T tracks
 *   of n_states stored states each: mean_f / mean_s [n_states][n][ld], cov_f / cov_s [n_states][n*n][ld] (distinct
 *   arrays), dt [n_states-1][ld], sog_rate / cog_rate [n_rates][ld] indexed by step / rate_repeat (the reference's
 *   np.repeat expansion, :287-292), noise [n_states-1][n][ld] unit normals in step order or NULL; status [T] or NULL.
 * ste_process_f64: one evaluation of the process model for T states, x_in / x_out [n][ld]. */
#define STE_MODEL_GEODETIC 0
#define STE_MODEL_GEODETIC_TURN 1
int ste_ukf_predict_n_f64(int32_t n, int32_t model, int32_t n_tracks, int64_t ld, const double *Q_host, double *x, double *P,
                          const double *dt, const double *sog_rate, const double *cog_rate, const double *noise,
                          double *sigma_prior, double *sigma_post, int32_t *status, void *stream);
int ste_ukf_update_n_f64(int32_t n, int32_t n_tracks, int64_t ld, const double *H_host, const double *R_host, double *x,
                         double *P, const double *z, const double *noise, int32_t *status, void *stream);
int ste_urtss_backward_n_f64(int32_t n, int32_t model, int32_t n_tracks, int64_t ld, int32_t n_states, int32_t rate_repeat,
                             int32_t n_rates, const double *Q_host, const double *mean_f, const double *cov_f, const double *dt,
                             const double *sog_rate, const double *cog_rate, const double *noise, double *mean_s,
                             double *cov_s, int32_t *status, void *stream);
int ste_process_f64(int32_t model, int32_t n, int32_t n_tracks, int64_t ld, const double *x_in, const double *dt,
                    const double *sog_rate, const double *cog_rate, double *x_out, void *stream);

/* Fleet path of the dimension-generic model (ABI 6): the n = 4 trio above for n = 5, STE_MODEL_GEODETIC_TURN.  Layout as
 * everywhere else (element (plane, t) at base[plane * ld + t]); matrices are row-major n x n planes.  The arithmetic is
 * that of ste_ukf_predict_n_f64 / ste_ukf_update_n_f64 / ste_urtss_backward_n_f64: every track is bit-identical to those
 * single-step kernels driven step by step.  No gating, full (not packed) covariances.  H, Q, R, P0: reference
 * UnscentedKalmanFilter.__init__ (unscented.py:20-74), row-major n x n in the first n*n entries; Q, R, P0 symmetric.
 * Q and R are shared by the tracks of a launch unless the _noise_ entry points below give each track its own
 * (SteNoiseN): such a track is bit-identical to the single-step kernels run with its matrices. */
typedef struct SteProblemN {
    int32_t n;             /* state dimension: 5                                            */
    int32_t model;         /* STE_MODEL_GEODETIC_TURN                                       */
    int32_t n_tracks;      /* T                                                             */
    int32_t max_steps;     /* N_max: filter steps of the longest track (states = N_max + 1) */
    int32_t max_obs;       /* rows available in the observation arrays                      */
    int32_t reserved;      /* must be 0                                                     */
    int64_t ld;            /* leading dimension of every SoA array (>= n_tracks)            */
    double H[64];
    double Q[64];
    double R[64];
    double P0[64];
} SteProblemN;

typedef struct SteInputsN {
    const double *x0;         /* [n][ld] initial state                                                   */
    const double *P0;         /* [n*n][ld] per-track prior covariance, or NULL -> SteProblemN.P0         */
    const double *dt;         /* [max_steps][ld] step lengths (hours)                                    */
    const uint8_t *upd_mask;  /* [max_steps][ld] 1 = step ends exactly on an observation time (forward) */
    const int32_t *n_steps;   /* [T] steps per track, or NULL -> max_steps for all                       */
    const double *z[8];       /* [max_obs][ld] observation rows 0 .. n-1; a NULL row is read as 0        */
    const double *sog_rate;   /* [max_obs][ld]                                                           */
    const double *cog_rate;   /* [max_obs][ld] or NULL (geodetic_dynamics_turn takes the turn rate from  */
                              /* the state)                                                              */
    const int32_t *rate_repeat; /* [T] backward-pass rate repeat per track (required by the backward)   */
    /* optional noise tapes of UNIT normals (NULL = zero noise), scaled by sqrt(diag Q) / sqrt(diag R)   */
    const double *noise_pred; /* [max_steps][n][ld]  unscented.py:198-202, row = step                    */
    const double *noise_upd;  /* [max_obs][n][ld]    unscented.py:232-236, row = update index            */
    const double *noise_bwd;  /* [max_steps][n][ld]  unscented.py:320-323, row = backward step           */
} SteInputsN;

typedef struct SteOutputsN {
    double *mean_f;      /* [max_steps+1][n][ld]   filtered means; row 0 = prior (kalman_filter.py:76)   */
    double *cov_f;       /* [max_steps+1][n*n][ld] filtered covariances                                  */
    double *mean_s;      /* smoothed, same shapes; distinct arrays (no in-place smoothing)              */
    double *cov_s;
    int32_t *status;     /* [T] OR-ed STE_STATUS_* (the forward pass overwrites, the backward ORs)      */
    int32_t *n_updates;  /* [T] observations assimilated incl. the initial one, or NULL                 */
} SteOutputsN;

/* KalmanFilterBase.run (kalman_filter.py:36-117) with UnscentedKalmanFilter.predict / update (unscented.py:144-265)
 * for T tracks of the five-state model: row 0 the prior, the initial update with observation 0, predict step s with
 * sog_rate / cog_rate at the current update index, an update with the next observation where upd_mask[s] is set
 * (more matches than max_obs rows: STE_STATUS_OBS_OVERRUN, update skipped).  n = 4 geodetic: ste_ukf_forward_f64. */
int ste_ukf_forward_n_f64(const SteProblemN *prob, const SteInputsN *in, SteOutputsN *out, void *stream);

/* UnscentedKalmanFilter.rts_step (unscented.py:267-351) for T ragged tracks: track t has n_steps[t] + 1 states and
 * reads rate[step / rate_repeat[t]]; reads mean_f / cov_f, writes mean_s / cov_s. */
int ste_urtss_backward_tracks_n_f64(const SteProblemN *prob, const SteInputsN *in, SteOutputsN *out, void *stream);

/* Per-track process and measurement noise for fleets that mix ship classes: the two passes above with each track's own
 * Q and R.  The planes are row-major n x n in the layout of SteInputsN.P0, element (i, j) of track t at
 * base[(i * n + j) * ld + t]; each replaces SteProblemN.Q / R for its track, noise tapes included (scaled by that
 * track's sqrt(diag Q) / sqrt(diag R)).  A NULL pointer, or noise == NULL, keeps the launch's shared matrix, and then the
 * call is the entry point above.  The backward pass reads Q_tracks only.  The planes must be symmetric: the library
 * cannot read device memory before the launch, so the caller checks it (the Python layer, batch_n.TrackBatchN, does).
 * These are separate entry points so that SteInputsN, and every binary built against it, stays as it was. */
typedef struct SteNoiseN {
    const double *Q_tracks;   /* [n*n][ld] per-track process noise, or NULL -> SteProblemN.Q     */
    const double *R_tracks;   /* [n*n][ld] per-track measurement noise, or NULL -> SteProblemN.R */
} SteNoiseN;
int ste_ukf_forward_noise_n_f64(const SteProblemN *prob, const SteInputsN *in, const SteNoiseN *noise, SteOutputsN *out,
                                void *stream);
int ste_urtss_backward_tracks_noise_n_f64(const SteProblemN *prob, const SteInputsN *in, const SteNoiseN *noise,
                                          SteOutputsN *out, void *stream);

/* UnscentedKalmanFilter.criterion_index and the denominator of update_lambda_factor
 * (unscented.py:389-483) for T filters: with y = z - x (not z - Hx, no angle wrap) and
 * S = H P H^T + R (prob->H, prob->R), gamma[t] = |y^T pinv(S) y| and denom[t] = y^T pinv(S) R pinv(S) y,
 * so that lambda' = lambda + (gamma - chi) / denom.  x [4][ld], P [16][ld], z [4][ld]; gamma, denom [T]. */
int ste_gate_terms_f64(const SteProblem *prob, const double *x, const double *P, const double *z,
                       double *gamma, double *denom, void *stream);

/* UnscentedKalmanFilter.compute_sigma_points (unscented.py:76-107), any n <= 8:
 * X[:, 0] = x, X[:, 1+i] = x + M[:, i], X[:, 1+n+i] = x - M[:, i], M = Re sqrtm(scale * P).
 * x [n][ld], P [n*n][ld], X [n*(2n+1)][ld] (plane = row*(2n+1) + point). */
int ste_sigma_points_f64(int32_t n, int32_t n_tracks, int64_t ld, double scale, const double *x,
                         const double *P, double *X, int32_t *status, void *stream);

/* geodetic_dynamics (non_linear_process.py:6-85) for T states: x_in/x_out [4][ld]. */
int ste_geodetic_f64(int32_t n_tracks, int64_t ld, const double *x_in, const double *dt,
                     const double *sog_rate, const double *cog_rate, double *x_out, void *stream);

/* Derived filter inputs from raw fixes for T tracks: ShipTrack.calculate_sog / calculate_cog /
 * calculate_sog_rate / calculate_cog_rate (ship_track.py:197-304) with the spherical pair
 * haversine_formula / heading (utils.py:75-147) and, when smooth_width > 1, the CLI's box smoothing
 * of SOG and COG (utils.py:150-172, main_cli.py:99-104: np.convolve(y, ones(w)/w, "same")).
 * geodesy STE_GEODESY_SPHERE: that spherical pair.  STE_GEODESY_WGS84: the reference's DEFAULT pair
 * geographiclib_distance / geographiclib_heading (utils.py:9-72), i.e. the WGS84 inverse geodesic of
 * the third-party geographiclib (>= 2.0, not vendored by the reference): restated here with
 * Vincenty's inverse formulae (same ellipsoid; agrees with the reference's one exact vector,
 * examples/cli_example/output_01203823_predictions.txt:1, to 8e-13 relative), including the
 * reference's "same point within 1e-8 degrees -> 0" guard; nearly antipodal legs, which Vincenty's
 * iteration does not resolve, give NaN.
 * lon, lat [max_obs][ld] degrees; dts [max_obs-1][ld] hours; n_obs [T] fixes per track or NULL;
 * outputs sog (km/h), cog (deg), sog_rate, cog_rate [max_obs][ld] (rows >= n_obs[t] are zeroed). */
#define STE_GEODESY_SPHERE 0
#define STE_GEODESY_WGS84 1
int ste_derive_inputs_f64(int32_t n_tracks, int32_t max_obs, int64_t ld, int32_t smooth_width, int32_t geodesy,
                          const double *lon, const double *lat, const double *dts, const int32_t *n_obs,
                          double *sog, double *cog, double *sog_rate, double *cog_rate, void *stream);

/* CSV rows -> columns for a whole file (ShipTrack.read_csv, ship_track.py:107-195, done for every ship at once):
 * `bytes` is the file as it sits on disk, copied to the device; row r is bytes[row_start[r] .. row_start[r+1] - 1)
 * (row_start has n_rows + 1 entries: the offset after each newline).  cols_host [8] (HOST array) gives the field index
 * of yr, mo, dy, hr, lat, lon, id and of the row-label column (-1: the file has no index column; label = row number).
 * Outputs [n_rows]: hours since 1970-01-01 00:00 of "yr-mo-dy hr:00" (the reference builds that string and parses it
 * with pandas; gaps between rows are differences of these), lat / lon (NaN for NA / empty), id_key (FNV-1a 64 of the id
 * text), id_int (its value when it is an integer literal), id_off / id_len (span of the id text inside the row),
 * label, flags (bit 0 bad date, 1 bad position, 2 id not an integer, 3 label not an integer, 4 lat / lon needs the
 * host's slow number path, 5 short row).  Fields may be double-quoted; no embedded quotes, commas or newlines. */
int ste_csv_parse_rows(const uint8_t *bytes, const int64_t *row_start, int64_t n_rows, const int32_t *cols_host, int64_t *hours,
                       double *lat, double *lon, uint64_t *id_key, int64_t *id_int, int32_t *id_off, int32_t *id_len,
                       int64_t *label, int32_t *flags, void *stream);

/* performance_metrics.rmse / abs_diff / cum_abs_diff (performance_metrics.py:4-58) of a state
 * estimate against the observations it assimilated, for T tracks in one launch.  For track t and
 * observation row r (rows with in->z[r] == NULL are skipped and left untouched), the pairs are
 * (x, xref) = (mean[s][r][t], z[r][u][t]) for u = 0 with s = 0 (the prior and the first fix) and,
 * for every later assimilated observation u, the state s that follows its update - the cadence is
 * the forward pass's (upd_mask / substeps, n_steps, max_obs).  No angle wrapping, as in the reference.
 * mean [max_steps+1][4][ld] (mean_f or mean_s); outputs, each [4][ld] or NULL: rmse = sqrt(mean of
 * squares), cum_abs = last element of cum_abs_diff (the sum of |x - xref|), max_abs = max of abs_diff;
 * abs_diff [max_obs][4][ld] or NULL receives every |x - xref|; n_pairs [T] or NULL the pair count. */
int ste_track_metrics_f64(const SteProblem *prob, const SteInputs *in, const double *mean, double *rmse,
                          double *cum_abs, double *max_abs, double *abs_diff, int32_t *n_pairs, void *stream);

/* ste_track_metrics_f64 for a tile of the five-state fleet path (ABI 7): the same pairs and reductions over observation
 * rows r < 5 (rows with in->z[r] == NULL are skipped and left untouched), the cadence from in->upd_mask (required) and
 * in->n_steps.  prob and in are checked as for ste_ukf_forward_n_f64 (x0, dt, sog_rate and the outputs are not read).
 * mean [max_steps+1][5][ld]; rmse, cum_abs, max_abs each [5][ld] or NULL; abs_diff [max_obs][5][ld] or NULL; n_pairs
 * [T] or NULL. */
int ste_track_metrics_n_f64(const SteProblemN *prob, const SteInputsN *in, const double *mean, double *rmse,
                            double *cum_abs, double *max_abs, double *abs_diff, int32_t *n_pairs, void *stream);

/* The CLI's text files for many ships at once: np.savetxt(path, X) with its defaults (fmt "%.18e", delimiter " ", newline
 * "\n"), as the reference CLI writes predictions, variances, dts and tracks (main_cli.py:146-167).  Every value is
 * formatted as CPython's "%.18e" % x (PyOS_double_to_string(x, 'e', 18): 19 significant digits, correctly rounded, ties
 * to even; "inf", "-inf", every NaN "nan"), followed by " " or, after a row's last column, "\n".
 *
 * A table is one file kind (say, the filtered means); an item is one ship.  Values are numbered item-major, then table,
 * row and column: segment g = item * n_tables + table holds values [value_start[g], value_start[g + 1]) (device,
 * n_items * n_tables + 1 entries, value_start[0] = 0, non-decreasing), rows of n_cols values.  Value (row r, column c)
 * of item i in table t is read from t.base[((r / t.row_div) * t.row_stride + t.plane[c]) * t.ld + t.track[i]], the usual
 * SoA layout (plane, track): the diagonal of a row-major n x n covariance is planes 0, n + 1, 2 (n + 1), ...; of the
 * packed 4 x 4 layout (STE_FLAG_PACKED_COV) planes 0, 4, 7, 9; row_div repeats source rows (the _dts file: dts /
 * substeps, each repeated substeps times).  value_start and track must only address rows and tracks the sources hold
 * (track[i] < n_tracks).
 *
 * ste_text_convert_f64: converts every value; digits [n_values] (the 19 significant digits as an integer), meta
 *   [n_values] (kind, sign, decimal exponent, separator) and length [n_values] (bytes of the field and its separator).
 * The caller forms end = inclusive scan of length (int64); the text of value v is out[end[v] - length[v], end[v]) and the
 *   file of segment g starts at the end of value value_start[g] - 1.
 * ste_text_write: writes the text of every value into out (device), which must hold STE_TEXT_MAX_VALUE_BYTES per value
 *   (the longest field, "-1.234567890123456789e-308", and its separator) whatever the total turns out to be. */
#define STE_TEXT_MAX_COLS 8
#define STE_TEXT_MAX_TABLES 8
#define STE_TEXT_MAX_VALUE_BYTES 27
typedef struct SteTextTable {
    const double *base;      /* source planes (device)                                          */
    const int32_t *track;    /* [n_items] column of item i in base (device)                     */
    int64_t ld;              /* leading dimension of base (>= n_tracks)                         */
    int32_t n_tracks;        /* columns of base                                                 */
    int32_t row_stride;      /* planes per source row (>= 1)                                    */
    int32_t row_div;         /* output row r reads source row r / row_div (>= 1)                */
    int32_t n_cols;          /* values per output row, 1 .. STE_TEXT_MAX_COLS                   */
    int32_t plane[STE_TEXT_MAX_COLS]; /* plane of column c within a source row, [0, row_stride) */
} SteTextTable;
int ste_text_convert_f64(const SteTextTable *tables, int32_t n_tables, int32_t n_items, const int64_t *value_start,
                         int64_t n_values, uint64_t *digits, int32_t *meta, int32_t *length, void *stream);
int ste_text_write(int64_t n_values, const uint64_t *digits, const int32_t *meta, const int64_t *end, uint8_t *out,
                   int64_t out_bytes, void *stream);

/* Test hook: evaluates the library's own fp64 elementary functions (csrc/ste_fastmath.cuh) on n
 * arguments.  kind 0 sincos(a), |a| <= 105615 -> (out0, out1); 1 atan2(a, b); 2 sqrt(a); 3 rsqrt(a); 4 1/a; 5 a/b;
 * 6 atan2(a, b) for b >= 0. */
int ste_probe_fastmath(int32_t kind, int32_t n, const double *a, const double *b, double *out0,
                       double *out1, void *stream);

/* Measurement helper: one block of `warps` warps runs `iters` rounds of n independent dependent
 * chains per thread, chains = 100 * mode + n with n in {1, 2, 4, 8}: mode 0 DFMA on registers,
 * 1 DFMA with constant-bank operands, 2 DMUL/DADD alternating, 3 DFMA followed by a compare +
 * select, 4 DFMA with three changing register sources (n in {4, 8}), 5 DMUL with two (n in {4, 8}).  cycles[0] (device int64) receives the clock64 span.  Gives the latency (warps = n = 1)
 * and the issue interval of the FP64 pipe for the instruction mixes the filter kernels issue. */
int ste_probe_fp64_latency(int32_t warps, int32_t iters, int32_t chains, double *sink,
                           long long *cycles, void *stream);

/* Measurement helper for the roofline report: runs `iters` dependent-free DFMA rounds on every
 * thread of `blocks` x `threads` and writes one double per thread to sink (device, blocks*threads).
 * FLOPs issued = 2 * 8 * iters * blocks * threads. */
int ste_probe_fp64_fma(int32_t blocks, int32_t threads, int32_t iters, double *sink, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* STE_UKF_H */
