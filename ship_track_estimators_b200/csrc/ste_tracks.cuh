// ste_tracks.cuh - the per-track time loops (forward filter, backward smoother).
//
// One call = one track, sequential in time.  The CUDA kernels in ste_ukf.cu call these with
// t = global thread index; the developer-side host sandbox (tools/host_emul) calls the very same
// code in a CPU loop to check numerical changes before GPU time is spent.
#pragma once
#include "ste_filter.cuh"

namespace ste {

template <typename T>
STE_DEV T min_(T a, T b) { return a < b ? a : b; }

// Asynchronous 8-byte global -> shared copy (LDGSTS): stages an input for later in the step
// without holding a register across the long sigma-point loop.  The host sandbox copies directly.
STE_DEV void stage_async(double *smem_dst, const double *gmem_src) {
#if defined(__CUDA_ARCH__)
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(gmem_src) : "memory");
#else
    *smem_dst = *gmem_src;
#endif
}
STE_DEV void stage_wait() {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.wait_all;" ::: "memory");
#endif
}

struct KernelArgs {
    SteProblem prob;
    SteInputs in;
    SteOutputs out;
};

// The scoring launch (ste_ukf_score_f64): the tile's arguments, the per-(candidate, track) sums and the candidate table,
// all in the kernel parameters.  Candidate blockIdx.y replaces prob.Q / prob.R; `out` is unused (zero).
struct KernelArgsScore : KernelArgs {
    SteScores scores;
    double Q[STE_MAX_CANDIDATES][16];
    double R[STE_MAX_CANDIDATES][16];
};

// Covariance storage: 16 planes per state (the full row-major 4x4 the reference returns) or, with
// STE_FLAG_PACKED_COV, only the 10 unique entries in SYM() order.  Both passes keep covariances
// exactly symmetric, so the packed form loses nothing; it cuts the state traffic by 30 %.
STE_DEV int cov_planes(bool packed) { return packed ? 10 : 16; }
STE_DEV int cov_plane(bool packed, int i, int j) { return packed ? SYM(i, j) : i * 4 + j; }

STE_DEV void store_state(double *mean, double *cov, int64_t ld, int64_t s, int t, bool packed,
                         const double (&x)[4], const double (&P)[10]) {
    // planes are consecutive in both layouts: plane k of a state is base + k * (ld * 8 bytes), one 32 x 32 + 64-bit
    // multiply-add per store (plane_ptr)
    const uint32_t ldb = (uint32_t)ld * 8u;
    double *m = mean + (s * 4) * ld + t;
#pragma unroll
    for (int r = 0; r < 4; ++r) STE_STORE_STREAM(plane_ptr(m, ldb, r), x[r]);
    double *c = cov + (s * cov_planes(packed)) * ld + t;
    if (packed) {
#pragma unroll
        for (int k = 0; k < 10; ++k) STE_STORE_STREAM(plane_ptr(c, ldb, k), P[k]);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) STE_STORE_STREAM(plane_ptr(c, ldb, i * 4 + j), P[SYM(i, j)]);
    }
}

STE_DEV void load_cov(const double *cov_state, int64_t ld, bool packed, double (&P)[10]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = i; j < 4; ++j) P[SYM(i, j)] = cov_state[cov_plane(packed, i, j) * ld];
}

STE_DEV void load_state(const double *mean, const double *cov, int64_t ld, int64_t s, int t, bool packed,
                        double (&x)[4], double (&P)[10]) {
    const double *m = mean + (s * 4) * ld + t;
#pragma unroll
    for (int r = 0; r < 4; ++r) x[r] = STE_LOAD_STREAM(m + r * ld);
    load_cov(cov + (s * cov_planes(packed)) * ld + t, ld, packed, P);
}

STE_DEV bool any_nonfinite(const double (&x)[4], const double (&P)[10]) {
    double acc = 0.0;
#pragma unroll
    for (int r = 0; r < 4; ++r) acc += x[r] * 0.0;
#pragma unroll
    for (int k = 0; k < 10; ++k) acc += P[k] * 0.0;
    return !(acc == 0.0);
}

// ------------------------------------------------------------------------------------------ //
// Forward filter: KalmanFilterBase.run (kalman_filter.py:36-117).
//
// The time loop is written as begin() / step(s) / end() on a small state object.
// INNOV: every update also stores its innovation statistics (struct Innov) into row u of the planes of `iv`.
// SCORE: the scoring form - candidate `cand` of `sa` supplies Q and R, nothing is stored per step (no states, no
// smoother tape, no gating planes: the robustification itself still runs) and the statistics of the updates are summed
// in update order, then written once per track into the candidate's row of sa->scores.
// PER_Q: the track's own process noise `q_track` (row-major 4x4, thread-local: forward_track loads it once, before the
// time loop) replaces the launch's Q.  Every read of Q (the predict's moments, the scaling of the noise tape) goes through
// Qm(), so such a track is bit-identical to a launch whose shared Q is its own.
// ------------------------------------------------------------------------------------------ //
template <bool POS_ONLY, bool GATING, bool INNOV = false, bool SCORE = false, bool PER_Q = false>
struct ForwardTrack {
    const KernelArgs &a;
    const SteInnovations *iv;
    const KernelArgsScore *sa;
    const int cand;
    const int t;
    const Scratch sc;
    const int64_t ld;
    const bool packed;
    int nt = 0, k_sub = 1;
    double x[4], P[10];
    int status = 0, ui = 0;
    // The smoother statistics are valid for the backward pass only if it would read the same
    // rates: it indexes them by step / rate_repeat (unscented.py:287-311), the filter by the
    // update index.  They agree on every regular step grid; a track where they do not is flagged
    // and smoothed by recomputation.
    int rep = 1, ri = 0, rc = 0;
    int sub_left = 1;   // predicts left until the next update when the cadence is "every k-th step"
    bool consistent = true, upd_next = false;
    double loglik_sum = 0.0, nis_sum = 0.0;   // SCORE: sums over the updates so far
    int dof_sum = 0;
    const double *const qt;   // PER_Q: the track's own Q

    STE_DEV ForwardTrack(const KernelArgs &args, int track, const Scratch &scratch, const SteInnovations *innov = nullptr,
                         const KernelArgsScore *score = nullptr, int candidate = 0, const double *q_track = nullptr)
        : a(args), iv(innov), sa(score), cand(candidate), t(track), sc(scratch), ld(args.prob.ld),
          packed((args.prob.flags & STE_FLAG_PACKED_COV) != 0), qt(q_track) {}

    // the process and measurement noise of the run: the tile's, (SCORE) the candidate's or (PER_Q) the track's own Q
    STE_DEV const double *Qm() const {
        if constexpr (SCORE) return sa->Q[cand];
        else if constexpr (PER_Q) return qt;
        else return a.prob.Q;
    }
    STE_DEV const double *Rm() const {
        if constexpr (SCORE) return sa->R[cand];
        else return a.prob.R;
    }

    // observation rows are staged into scratch a whole predict ahead of their use
    // row u of a [row][track] input array for this track: base + t, then one 32 x 32 + 64-bit multiply-add (plane_ptr)
    STE_DEV const double *row_ptr(const double *base, int u) const { return plane_ptr(base + t, (uint32_t)ld * 8u, (uint32_t)u); }
    STE_DEV void stage_obs(int u) const {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            if ((!POS_ONLY || r < 2) && a.in.z[r]) stage_async(&sc.at(kScratchObs + r), row_ptr(a.in.z[r], u));
        }
    }
    // Inputs of step s (dt, the two rates, the observation of its update) are staged into shared
    // scratch with cp.async one whole step ahead: no register is held across the sigma-point loop
    // and the DRAM latency hides behind ~4000 instructions of the previous step.
    STE_DEV void stage_step(int s, int rate_index) const {
        stage_async(&sc.at(kScratchIn + 0), row_ptr(a.in.dt, s));
        stage_async(&sc.at(kScratchIn + 1), row_ptr(a.in.sog_rate, rate_index));
        stage_async(&sc.at(kScratchIn + 2), row_ptr(a.in.cog_rate, rate_index));
    }
    // does step s end on an observation?  (called once per step, in order: s = 0, 1, 2, ...)
    STE_DEV bool step_updates(int s) {
        if (a.in.upd_mask) return a.in.upd_mask[(int64_t)s * ld + t] != 0;
        if (--sub_left > 0) return false;   // (s + 1) % k_sub == 0 without the division
        sub_left = k_sub;
        return true;
    }

    STE_DEV void assimilate(int u) {
        // a per-track measurement covariance (SteInputs.R_tracks: ships with different sensors) replaces the
        // shared R; only the generic update reads a full 4x4 R
        const double *Rp = Rm();
        double Rt[16];
        if constexpr (!POS_ONLY) {
            if (a.in.R_tracks) {
#pragma unroll
                for (int k = 0; k < 16; ++k) Rt[k] = a.in.R_tracks[k * ld + t];
                Rp = Rt;
            }
        }
        const Model model{a.prob.H, Qm(), Rp};
        double z[4], un[4];
        stage_wait();
#pragma unroll
        for (int r = 0; r < 4; ++r) z[r] = sc.at(kScratchObs + r);
        const double *noise = nullptr;
        if (a.in.noise_upd) {
#pragma unroll
            for (int r = 0; r < 4; ++r) un[r] = a.in.noise_upd[((int64_t)u * 4 + r) * ld + t];
            noise = un;
        }
        int it;
        double lam, rs;
        Innov st;
        if (POS_ONLY)
            ukf_update_position<GATING, INNOV || SCORE>(x, P, model, z, noise, a.prob.gate_chi, a.prob.gate_max_iter, status, it, lam, rs, &st);
        else
            ukf_update_generic<GATING, INNOV || SCORE>(x, P, model, z, noise, a.prob.gate_chi, a.prob.gate_max_iter, status, it, lam, rs, &st);
        if (GATING && !SCORE) {
            if (a.out.gate_iters) a.out.gate_iters[(int64_t)u * ld + t] = (uint8_t)min_(it, 255);
            if (a.out.gate_lambda) a.out.gate_lambda[(int64_t)u * ld + t] = lam;
            if (a.out.gate_scale) a.out.gate_scale[(int64_t)u * ld + t] = rs;
        }
        if constexpr (INNOV) {
            const int64_t row = (int64_t)u * ld + t;
            iv->nis[row] = st.nis;
            iv->loglik[row] = -0.5 * fma((double)st.rank, kLog2Pi, st.nis + st.log_pdet);
            iv->rank[row] = (uint8_t)st.rank;
        }
        if constexpr (SCORE) {   // the expression the innovation planes store, added in update order
            loglik_sum += -0.5 * fma((double)st.rank, kLog2Pi, st.nis + st.log_pdet);
            nis_sum += st.nis;
            dof_sum += st.rank;
        }
    }

    STE_DEV void begin() {
        nt = a.in.n_steps ? min_(a.in.n_steps[t], a.prob.max_steps) : a.prob.max_steps;
        k_sub = a.prob.substeps > 0 ? a.prob.substeps : 1;
        sub_left = k_sub;
#pragma unroll
        for (int r = 0; r < 4; ++r) x[r] = a.in.x0[r * ld + t];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = i; j < 4; ++j)
                P[SYM(i, j)] = a.in.P0 ? a.in.P0[(i * 4 + j) * ld + t] : a.prob.P0[i * 4 + j];
        if constexpr (!SCORE) store_state(a.out.mean_f, a.out.cov_f, ld, 0, t, packed, x, P);  // the prior (kalman_filter.py:76-77)
#pragma unroll
        for (int r = 0; r < 4; ++r) sc.at(kScratchObs + r) = 0.0;   // absent rows read as 0
        stage_obs(0);
        rep = a.in.rate_repeat ? a.in.rate_repeat[t] : a.prob.rate_repeat;
        rep = rep > 0 ? rep : 1;
        if (nt > 0) {
            stage_step(0, 0);
            upd_next = step_updates(0);
        }
        assimilate(0);   // kalman_filter.py:81 (waits for the staged copies, including step 0's inputs)
    }

    STE_DEV void step(int s) {
        const bool upd = upd_next;
        const double dt = sc.at(kScratchIn + 0), sr = sc.at(kScratchIn + 1), cr = sc.at(kScratchIn + 2);
        consistent &= (min_(ri, a.prob.max_obs - 1) == ui);
        if (++rc == rep) {
            rc = 0;
            ++ri;
        }
        const bool advance = upd && (ui + 1 < a.prob.max_obs);
        if (upd && !advance) status |= STE_STATUS_OBS_OVERRUN;
        // stage what this step's update and the next step's predict will read
        if (advance) stage_obs(ui + 1);
        if (s + 1 < nt) {
            stage_step(s + 1, ui + (advance ? 1 : 0));
            upd_next = step_updates(s + 1);
        }
        double *stats = (!SCORE && a.out.smooth_stats) ? a.out.smooth_stats + ((int64_t)s * kStatsPlanes) * ld + t : nullptr;
        double e[4] = {0.0, 0.0, 0.0, 0.0};
        if (a.in.noise_pred) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
                e[r] = a.in.noise_pred[((int64_t)s * 4 + r) * ld + t] * sqrt(Qm()[r * 5]);
        }
        ukf_predict(x, P, Qm(), dt, sr, cr, e, status, sc, nullptr, nullptr, stats, ld, !(a.prob.flags & STE_FLAG_LONG_STEPS),
                    a.in.noise_pred != nullptr);
        // more matched update times than observation rows: the reference raises IndexError here
        // (kalman_filter.py:101-108); the track is flagged and the update skipped, nothing is re-read
        if (advance) assimilate(++ui);
        else stage_wait();   // the next step's inputs must have landed before they are read
        if constexpr (!SCORE) store_state(a.out.mean_f, a.out.cov_f, ld, s + 1, t, packed, x, P);
    }

    STE_DEV void end() {
        if (any_nonfinite(x, P)) status |= STE_STATUS_NONFINITE;
        if constexpr (SCORE) {
            const SteScores &o = sa->scores;
            const int64_t row = (int64_t)cand * o.ld_out + t;
            o.loglik[row] = loglik_sum;
            o.nis[row] = nis_sum;
            o.dof[row] = dof_sum;
            o.n_updates[row] = ui + 1;
            o.status[row] = status;
        } else {
            if (a.out.smooth_stats && !consistent) status |= STE_STATUS_SMOOTH_RECOMPUTE;
            a.out.status[t] = status;
            if (a.out.n_updates) a.out.n_updates[t] = ui + 1;
        }
    }
};

template <bool POS_ONLY, bool GATING, bool INNOV = false, bool SCORE = false, bool PER_Q = false>
STE_DEV void forward_track(const KernelArgs &a, const int t, const Scratch &sc, const SteInnovations *iv = nullptr,
                           const KernelArgsScore *sa = nullptr, int cand = 0, const double *q_planes = nullptr) {
    // PER_Q: the track's Q from the planes q_planes [16][ld] (the layout of SteInputs.P0 / R_tracks)
    double Qt[PER_Q ? 16 : 1];
    if constexpr (PER_Q) {
#pragma unroll
        for (int k = 0; k < 16; ++k) Qt[k] = q_planes[k * a.prob.ld + t];
    }
    ForwardTrack<POS_ONLY, GATING, INNOV, SCORE, PER_Q> f(a, t, sc, iv, sa, cand, PER_Q ? Qt : nullptr);
    f.begin();
#if defined(STE_STEP_SYNC) && defined(__CUDA_ARCH__)
    // experiment: the warps of a block start every step together (instruction-cache locality); ragged lengths are safe,
    // the loop runs while any thread of the block has a step left
#pragma unroll 1
    for (int s = 0; __syncthreads_or(s < f.nt); ++s) {
        if (s < f.nt) f.step(s);
    }
#else
#pragma unroll 1
    for (int s = 0; s < f.nt; ++s) f.step(s);
#endif
    f.end();
}

// ------------------------------------------------------------------------------------------ //
// Backward smoother: UnscentedKalmanFilter.rts_step (unscented.py:267-351).
// PER_Q: the track's own Q (planes as in ForwardTrack) wherever the step reads Q - the scaling of the noise tape, the
// speed / course blocks of the predicted covariance rebuilt from the tape, and the recomputed moments.  The forward pass
// put the same track's Q into the tape's position block, so both passes must be given the same planes.
// ------------------------------------------------------------------------------------------ //
STE_DEV void prefetch_l2(const void *p) {
#if defined(__CUDA_ARCH__)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#else
    (void)p;
#endif
}

template <bool PER_Q = false>
struct BackwardTrack {
    const KernelArgs &a;
    const int t;
    Scratch sc;
    const int64_t ld;
    const bool packed;
    int nt = 0, rep = 1, status = 0;
    // Statistics stored by the forward pass replace the sigma-point recomputation for every step
    // but step 0: state 0 is the PRIOR (kalman_filter.py:76-81), which the filter never predicted
    // from (it predicted from the prior's update), so its statistics do not exist.
    bool use_stats = false, bad = false;
    const double *const qt;   // PER_Q: the track's own Q

    STE_DEV BackwardTrack(const KernelArgs &args, int track, const Scratch &scratch, const double *q_track = nullptr)
        : a(args), t(track), sc(scratch), ld(args.prob.ld), packed((args.prob.flags & STE_FLAG_PACKED_COV) != 0), qt(q_track) {}

    STE_DEV const double *Qm() const {
        if constexpr (PER_Q) return qt;
        else return a.prob.Q;
    }

    STE_DEV void begin() {
        nt = a.in.n_steps ? min_(a.in.n_steps[t], a.prob.max_steps) : a.prob.max_steps;
        rep = a.in.rate_repeat ? a.in.rate_repeat[t] : a.prob.rate_repeat;
        rep = rep > 0 ? rep : 1;
        // the last state is untouched by the smoother (:297); it seeds the carried (xs, Ps)
        double xs[4], Ps[10];
        load_state(a.out.mean_f, a.out.cov_f, ld, nt, t, packed, xs, Ps);
        if (a.out.mean_s != a.out.mean_f || a.out.cov_s != a.out.cov_f)
            store_state(a.out.mean_s, a.out.cov_s, ld, nt, t, packed, xs, Ps);
#pragma unroll
        for (int r = 0; r < 4; ++r) sc.at(kScratchXs + r) = xs[r];
#pragma unroll
        for (int k = 0; k < 10; ++k) sc.at(kScratchPs + k) = Ps[k];
        use_stats = a.out.smooth_stats && !(a.out.status[t] & STE_STATUS_SMOOTH_RECOMPUTE);
    }

    // Pull what step(step) will read from the statistics path towards L2 (no register, no scratch).
    STE_DEV void prefetch_stats_step(int step) const {
        const double *mf = a.out.mean_f + ((int64_t)step * 4) * ld + t;
        const double *cf = a.out.cov_f + ((int64_t)step * cov_planes(packed)) * ld + t;
        const double *st = a.out.smooth_stats + ((int64_t)step * kStatsPlanes) * ld + t;
#pragma unroll
        for (int r = 0; r < 4; ++r) prefetch_l2(mf + r * ld);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = i; j < 4; ++j) prefetch_l2(cf + cov_plane(packed, i, j) * ld);
#pragma unroll
        for (int k = 0; k < kStatsPlanes; ++k) prefetch_l2(st + k * ld);
    }

    STE_DEV void step(int step) {
        const double *mf = a.out.mean_f + ((int64_t)step * 4) * ld + t;
        const double *cf = a.out.cov_f + ((int64_t)step * cov_planes(packed)) * ld + t;
        double xs[4], Ps[10];
        double e[4] = {0.0, 0.0, 0.0, 0.0};
        if (a.in.noise_bwd) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
                e[r] = a.in.noise_bwd[((int64_t)step * 4 + r) * ld + t] * sqrt(Qm()[r * 5]);
        }
        bool done = false;
#ifndef STE_BWD_PREFETCH
#define STE_BWD_PREFETCH 1
#endif
        // The tape pass is bound by memory latency at its 8 warps per SM (29 loads in flight per thread and step):
        // pulling the NEXT step's 29 lines towards L2 now, without registers, turns its DRAM round trip into an L2 hit.
        if (STE_BWD_PREFETCH && use_stats && step > STE_BWD_PREFETCH) prefetch_stats_step(step - STE_BWD_PREFETCH);   // distance in steps
        if (use_stats && step > 0)
            done = urtss_step_from_stats(mf, cf, packed, a.out.smooth_stats + ((int64_t)step * kStatsPlanes) * ld + t, ld, Qm(),
                                         e, xs, Ps, status, sc, (unsigned)a.prob.reserved);
        if (!done) {
            double xf[4], s1[4], Pb[10];
#pragma unroll
            for (int r = 0; r < 4; ++r) xf[r] = mf[r * ld];
            const double dt = a.in.dt[(int64_t)step * ld + t];
            const int ri = min_(step / rep, a.prob.max_obs - 1);
            const double sr = a.in.sog_rate[(int64_t)ri * ld + t];
            const double cr = a.in.cog_rate[(int64_t)ri * ld + t];
            {
                double Pf[10];
                load_cov(cf, ld, packed, Pf);
                if (step > 0) {   // pull the next (earlier) state towards L2 while this step computes
#pragma unroll
                    for (int r = 0; r < 4; ++r) prefetch_l2(mf + (r - 4) * ld);
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = i; j < 4; ++j) prefetch_l2(cf + (cov_plane(packed, i, j) - cov_planes(packed)) * ld);
                    prefetch_l2(a.in.dt + (int64_t)(step - 1) * ld + t);
                }
                urtss_moments<PER_Q>(xf, Pf, Qm(), dt, sr, cr, s1, Pb, status, sc);
            }
            double Pf[10];   // again (L2-resident) rather than held across the sigma-point loop
            load_cov(cf, ld, packed, Pf);
            urtss_gain(xf, Pf, s1, Pb, e, xs, Ps, status, sc);
        }
        store_state(a.out.mean_s, a.out.cov_s, ld, step, t, packed, xs, Ps);
        bad |= any_nonfinite(xs, Ps);
    }

    STE_DEV void end() {
        if (bad) status |= STE_STATUS_NONFINITE;
        a.out.status[t] |= status;
    }
};

template <bool PER_Q = false>
STE_DEV void backward_track(const KernelArgs &a, const int t, const Scratch &sc, const double *q_planes = nullptr) {
    double Qt[PER_Q ? 16 : 1];   // as forward_track
    if constexpr (PER_Q) {
#pragma unroll
        for (int k = 0; k < 16; ++k) Qt[k] = q_planes[k * a.prob.ld + t];
    }
    BackwardTrack<PER_Q> g(a, t, sc, PER_Q ? Qt : nullptr);
    g.begin();
#pragma unroll 1
    for (int step = g.nt - 1; step >= 0; --step) g.step(step);
    g.end();
}

}  // namespace ste
