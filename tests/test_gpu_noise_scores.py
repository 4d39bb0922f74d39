"""GPU: noise-candidate scores (``BatchedUKF.score`` / ``BatchedUKFN.score``, ``ste_ukf_score_f64`` /
``ste_ukf_score_n_f64``) and the maximum-likelihood choice of ``tuning.fit_noise``.

The oracle is the validated innovations path: for every candidate, a filter built with that candidate's ``Q`` / ``R`` runs
``run(b, smoother=False, innovations=True)``, and its per-update ``loglik`` / ``nis`` planes summed in update order must
equal the scores bit for bit, with ``dof``, ``n_updates`` and ``status`` equal."""
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import ukf_numpy as O
from test_gpu_innovations import H_DENSE, H_POS, P_DEF, Q_DEF, R_DENSE, R_GATE, R_POS, _fleet4, _tapes4

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, scope="module")
def _release_cached_blocks():
    yield
    import torch

    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _sums(res):
    """Per-column sums of an innovations run, in update order: what the scores must equal bit for bit."""
    n_upd = res.n_updates.cpu().numpy()
    L, N, rank = res.loglik.cpu().numpy(), res.nis.cpu().numpy(), res.innov_rank.cpu().numpy().astype(np.int64)
    cols = range(len(n_upd))
    return {"loglik": np.array([np.cumsum(L[: n_upd[t], t])[-1] for t in cols]),
            "nis": np.array([np.cumsum(N[: n_upd[t], t])[-1] for t in cols]),
            "dof": np.array([rank[: n_upd[t], t].sum() for t in cols]), "n_updates": n_upd, "status": res.status.cpu().numpy()}


def _assert_equal(score, c, ref, where):
    for key in ("loglik", "nis"):
        got = score[key][c].cpu().numpy()
        assert np.array_equal(got, ref[key], equal_nan=True), (where, c, key, float(np.nanmax(np.abs(got - ref[key]))))
    for key in ("dof", "n_updates", "status"):
        assert np.array_equal(score[key][c].cpu().numpy(), ref[key]), (where, c, key)


def _check_against_runs(make_engine, b, cands, where):
    """Score every candidate in one call and compare each with its own innovations run."""
    engine = make_engine(*cands[0])
    score = engine.score(b, cands)
    assert all(v.shape == (len(cands), b.n_tracks) for v in score.values())
    for c, (Qc, Rc) in enumerate(cands):
        ref = _sums(make_engine(Qc, Rc).run(b, smoother=False, innovations=True))
        _assert_equal(score, c, ref, where)
    return score


# --------------------------------------------------------------------------- #
# n = 4                                                                       #
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("long_steps", [False, True])
@pytest.mark.parametrize("case", ["position", "force_generic", "dense", "gated"])
def test_n4_scores_equal_the_innovation_runs(case, long_steps, cuda, native_lib):
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.tuning import noise_grid

    gating = case == "gated"
    H, R = {"position": (H_POS, R_POS), "force_generic": (H_POS, R_POS), "dense": (H_DENSE, R_DENSE), "gated": (H_POS, R_GATE)}[case]
    tracks, dts = _fleet4(80, 36, seed=900 + len(case), k=2, outliers=0.05 if gating else 0.0)
    noise = None if gating else _tapes4(tracks, dts, 21)   # tapes are scaled by each candidate's own sqrt(diag Q / R)
    b = TrackBatch.from_tracks(tracks, dts, device=cuda, noise=noise)
    cands = noise_grid(Q_DEF, R, (0.5, 1.0, 4.0), (0.25, 1.0, 4.0))

    def make(Qc, Rc):
        return BatchedUKF(H, Qc, Rc, P_DEF, gating=gating, force_generic=case in ("force_generic", "dense"), packed_cov=True,
                          long_steps=long_steps)

    _check_against_runs(make, b, cands, (case, long_steps))
    if gating:   # the displaced fixes were robustified
        res = make(*cands[4]).run(b, smoother=False)
        assert int(res.gate_iters.sum()) > 0


def test_n4_forty_candidates_chunked_and_split(cuda, native_lib):
    """40 candidates, position-only and generic R interleaved: two variant groups, the larger one over two launches and
    neither contiguous.  Every candidate equals its own single-candidate score, and two of them their innovation runs.
    The tile is in the cadence form (every second step updates, no upd_mask)."""
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.synthetic import make_tracks

    b = TrackBatch.from_synthetic(make_tracks(640, 40, seed=950, device="cpu", dts_choices=(1.0, 2.0)), substeps=2,
                                  need_rows=(True, True, True, True)).to(cuda)
    assert b.upd_mask is None
    cands = []
    for c in range(40):
        s = 0.25 * (1 + c % 9)
        R = np.diag([s * 1e-3, s * 1e-3, 0.0, 0.0]) if c % 7 != 3 else np.diag([s * 1e-3, s * 1e-3, 0.5 * s, 4.0])
        cands.append((Q_DEF * (1 + c // 9), R))
    ukf = BatchedUKF(H_POS, Q_DEF, R_POS, P_DEF)
    assert ukf.model.position_only()
    score = ukf.score(b, cands)
    for c, cand in enumerate(cands):
        one = ukf.score(b, [cand])
        for key in score:
            assert np.array_equal(score[key][c].cpu().numpy(), one[key][0].cpu().numpy(), equal_nan=True), (c, key)
    for c in (3, 38):   # a generic and a position-only candidate of the second chunk
        ref = _sums(BatchedUKF(H_POS, cands[c][0], cands[c][1], P_DEF).run(b, smoother=False, innovations=True))
        _assert_equal(score, c, ref, "forty")


# --------------------------------------------------------------------------- #
# n = 5                                                                       #
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("k,tapes", [(1, False), (2, False), (1, True)])
def test_n5_scores_equal_the_innovation_runs(k, tapes, cuda, native_lib):
    from test_gpu_fleet_n5 import H5, P5, Q5, R5, _fleet
    from test_gpu_fleet_n5_noise import _tapes

    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.tuning import noise_grid

    tracks, dts, x0 = _fleet(100, 30, seed=960 + k, ks=(k,), nobs_min=4)
    b = TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda, noise=_tapes(tracks, dts, 31) if tapes else None)
    cands = noise_grid(Q5, R5, (0.5, 2.0), (0.25, 1.0, 4.0))
    _check_against_runs(lambda Qc, Rc: BatchedUKFN(H5, Qc, Rc, P5), b, cands, (k, tapes))


def test_fit_noise_per_track_over_fleet_tiles(cuda, native_lib):
    """fit_noise(per="track") over several tiles returns, in the caller's order, the argmax of each track's summed
    log-likelihood over one innovations run per candidate."""
    from test_gpu_fleet_n5 import H5, P5, Q5, R5, _fleet

    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.tuning import fit_noise, noise_grid

    tracks, dts, x0 = _fleet(150, 30, seed=970, nobs_min=3)
    tiles = TrackBatchN.fleet_tiles(tracks, dts, x0=x0, device=cuda, state_budget=1500, granule=8)
    assert len(tiles) > 1
    cands = noise_grid(Q5, R5, (0.25, 1.0, 4.0), (0.1, 1.0, 10.0))
    fit = fit_noise(BatchedUKFN(H5, Q5, R5, P5), tiles, cands, per="track")
    whole = TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda)
    cols = np.arange(len(tracks)) if whole.order is None else np.argsort(whole.order)   # caller i -> column
    table = np.stack([_sums(BatchedUKFN(H5, Qc, Rc, P5).run(whole, smoother=False, innovations=True))["loglik"][cols]
                      for Qc, Rc in cands])
    want = np.argmax(np.where(np.isfinite(table), table, -np.inf), axis=0)
    assert np.array_equal(fit["loglik"], table, equal_nan=True)
    assert fit["best"].tolist() == want.tolist()
    for i, c in enumerate(want):
        assert fit["Q"][i] is cands[c][0] and fit["R"][i] is cands[c][1]
    # the per-track choice feeds the per-track noise planes directly
    chosen = TrackBatchN.fleet_tiles(tracks, dts, x0=x0, device=cuda, Q=fit["Q"], R=fit["R"])
    assert len(chosen) >= 1 and all(t.Q is not None and t.R is not None for t in chosen)


# --------------------------------------------------------------------------- #
# recovery of the true measurement noise                                      #
# --------------------------------------------------------------------------- #
Q_TRUE = np.diag([1e-4, 1e-4, 0.2, 4.0])
R_TRUE = 0.05 ** 2   # deg^2 on longitude and latitude
P_TRUE = np.diag([R_TRUE, R_TRUE, 4.0, 100.0])
R_SCALES = (0.25, 0.5, 1.0, 2.0, 4.0)


def _recovery_fleet(T, m, seed):
    """A correctly specified fleet: the truth stepped by the filter's own model (geodetic_dynamics at zero rates, hourly)
    plus process noise Q_TRUE, position fixes with noise R_TRUE.  Returns the tracks and their true initial states."""
    rng = np.random.default_rng(seed)
    tracks, x0 = [], []
    for _ in range(T):
        x = np.array([rng.uniform(-40, 40), rng.uniform(-50, 50), rng.uniform(10, 30), rng.uniform(0, 360)])
        states = [x]
        for _ in range(m - 1):
            x = O.geodetic_dynamics(x, 1.0, 0.0, 0.0) + rng.multivariate_normal(np.zeros(4), Q_TRUE)
            states.append(x)
        z = np.array(states).T
        z[:2] += rng.normal(scale=np.sqrt(R_TRUE), size=(2, m))
        tracks.append(SimpleNamespace(dts=np.ones(m - 1), z=z, sog_rate=np.zeros(m), cog_rate=np.zeros(m)))
        x0.append(states[0])
    return tracks, x0


def test_recovery_picks_the_true_r(cuda, native_lib):
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.tuning import fit_noise, noise_grid

    tracks, x0 = _recovery_fleet(64, 60, seed=900)
    b = TrackBatch.from_tracks(tracks, [tr.dts for tr in tracks], x0=x0, device=cuda)
    R0 = np.diag([R_TRUE, R_TRUE, 0.0, 0.0])
    cands = noise_grid(Q_TRUE, R0, (1.0,), R_SCALES)
    fit = fit_noise(BatchedUKF(H_POS, Q_TRUE, R0, P_TRUE), b, cands, per="fleet")
    assert fit["best"] == R_SCALES.index(1.0), fit["loglik"]
    assert len(fit["excluded"]) == 0 and np.array_equal(fit["R"], R0)
