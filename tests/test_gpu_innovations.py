"""GPU: per-update innovation statistics of the forward passes (``allocate(..., innovations=True)``,
``ste_ukf_forward_innov_f64`` / ``ste_ukf_forward_innov_n_f64``) - every existing output bit-identical with and without
the planes, nis / loglik / rank against a numpy reference built from the oracle's predict / update, the planes following
their tracks through the packing order, ``run_many`` (also partitioned) and noise selection by maximum likelihood."""
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import ukf_numpy as O

pytestmark = pytest.mark.gpu

H_POS = np.diag([1.0, 1.0, 0.0, 0.0])
R_POS = np.diag([1e-3, 1e-3, 0.0, 0.0])
Q_DEF = np.diag([1e-2, 1e-2, 1e-4, 1e-4])
P_DEF = np.eye(4)
# a dense measurement matrix and a full R: the generic update with every row and column in use
H_DENSE = np.array([[1.0, 0.1, 0.0, 0.0], [0.05, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.02], [0.0, 0.0, 0.01, 1.0]])
R_DENSE = np.array([[2e-3, 5e-4, 0.0, 0.0], [5e-4, 1e-3, 0.0, 0.0], [0.0, 0.0, 0.5, 0.1], [0.0, 0.0, 0.1, 4.0]])
R_GATE = np.diag([0.05, 0.05, 0.0, 0.0])
LOG2PI = np.log(2.0 * np.pi)
KEYS4 = ("means", "covs", "means_s", "covs_s", "status", "n_updates", "gate_iters", "gate_lambda", "gate_scale")


@pytest.fixture(autouse=True, scope="module")
def _release_cached_blocks():
    yield
    import torch

    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


# --------------------------------------------------------------------------- #
# numpy reference                                                             #
# --------------------------------------------------------------------------- #
def _stats(S, y):
    """nis, loglik and rank of one update from numpy's eigh with pinv's cutoff."""
    w, V = np.linalg.eigh(S)
    keep = np.abs(w) > 1e-15 * np.max(np.abs(w))
    nis = float(y @ ((V[:, keep] / w[keep]) @ V[:, keep].T) @ y)
    with np.errstate(invalid="ignore"):
        lpd = float(np.sum(np.log(w[keep])))
    r = int(keep.sum())
    return nis, -0.5 * (nis + lpd + r * LOG2PI), r


def _ref4(tr, dt_array, x0, H, Q, R, P0, gating=False, noise=None, pos=False):
    """kalman_filter.py:36-117 through the oracle's predict / update, with the statistics of every update formed from
    the state it receives (R scaled by the robustification, z after the noise draw)."""
    src = O.TapeNoise(**noise) if noise else O.ZeroNoise()
    x, P = np.array(x0, dtype=np.float64), np.array(P0, dtype=np.float64)
    mask = O.update_mask(dt_array, tr.dts)
    out = []

    def assimilate(x, P, zcol):
        Ruse = O.check_robustness(x, zcol, P, H, R)[0] if gating else R
        z = zcol + src.draw("upd", np.sqrt(np.diag(Ruse)))
        y = z - H @ x
        y[3] = O.wrap180(y[3])
        S = H @ P @ H.T + Ruse
        rows = [0, 1] if pos else [0, 1, 2, 3]
        out.append(_stats(S[np.ix_(rows, rows)], y[rows]))
        return O.update(x, P, H, Ruse, z, O.ZeroNoise())

    ui = 0
    x, P = assimilate(x, P, tr.z[:, 0])
    for step, dt in enumerate(dt_array):
        x, P, _, _ = O.predict(x, P, Q, dt, tr.sog_rate[ui], tr.cog_rate[ui], src)
        if mask[step]:
            ui += 1
            x, P = assimilate(x, P, tr.z[:, ui])
    return np.array(out)


def _ref5(tr, dt_array, x0, H, Q, R, P0):
    from _oracle_n5 import predict

    x, P = np.array(x0, dtype=np.float64), np.array(P0, dtype=np.float64)
    mask = O.update_mask(dt_array, tr.dts)
    out = []

    def assimilate(x, P, z):
        y = z - H @ x
        y[3] = O.wrap180(y[3])
        out.append(_stats(H @ P @ H.T + R, y))
        return O.update(x, P, H, R, z.copy(), O.ZeroNoise())

    ui = 0
    x, P = assimilate(x, P, tr.z[:, 0])
    for step, dt in enumerate(dt_array):
        x, P = predict(x, P, Q, dt, tr.sog_rate[ui])
        if mask[step]:
            ui += 1
            x, P = assimilate(x, P, tr.z[:, ui])
    return np.array(out)


def _assert_stats(got, ref, where):
    assert len(got["nis"]) == len(ref), where
    for key, col in (("nis", 0), ("loglik", 1)):
        err = np.abs(got[key] - ref[:, col]) / np.maximum(1.0, np.abs(ref[:, col]))
        assert float(np.max(err)) <= 1e-9, (where, key, float(np.max(err)))
    assert np.array_equal(got["innov_rank"], ref[:, 2].astype(np.int32)), where


def _assert_untouched(res):
    """Rows at or beyond a track's n_updates keep their allocation values (NaN, rank 0)."""
    import torch

    rows = torch.arange(res.nis.shape[0], device=res.nis.device)[:, None]
    beyond = rows >= res.n_updates.to(torch.int64)[None, :]
    assert bool(res.nis[beyond].isnan().all()) and bool(res.loglik[beyond].isnan().all())
    assert bool((res.innov_rank[beyond] == 0).all())
    assert not bool(res.nis[~beyond].isnan().any())


# --------------------------------------------------------------------------- #
# fleets                                                                      #
# --------------------------------------------------------------------------- #
def _fleet4(T, nobs_max, seed, k, outliers=0.0, nobs_min=5):
    from ship_track_estimators_b200.synthetic import make_tracks
    from ship_track_estimators_b200.utils import generate_dts

    syn = make_tracks(T, nobs_max, seed=seed, device="cpu", nobs_min=nobs_min, dts_choices=(1.0, 2.0, 3.0), outlier_frac=outliers)
    tracks, dts = [], []
    for t in range(T):
        m = int(syn.nobs[t])
        z = np.stack([syn.lon[:m, t].numpy(), syn.lat[:m, t].numpy(), syn.sog[:m, t].numpy(), syn.cog[:m, t].numpy()])
        tracks.append(SimpleNamespace(dts=syn.dts[: m - 1, t].numpy().copy(), z=z, sog_rate=syn.sog_rate[:m, t].numpy().copy(),
                                      cog_rate=syn.cog_rate[:m, t].numpy().copy()))
        dts.append(generate_dts(tracks[-1].dts, k))
    return tracks, dts


def _tapes4(tracks, dts, seed):
    rng = np.random.default_rng(seed)
    return [dict(pred=rng.normal(size=(len(d), 4)), upd=rng.normal(size=(tr.z.shape[1], 4)), bwd=rng.normal(size=(len(d), 4)))
            for tr, d in zip(tracks, dts)]


def _same(a, b, keys, where):
    for key in keys:
        if key in a or key in b:
            assert np.array_equal(a[key], b[key]), (where, key)


# --------------------------------------------------------------------------- #
# n = 4                                                                       #
# --------------------------------------------------------------------------- #
@pytest.mark.parametrize("generic", [False, True])
@pytest.mark.parametrize("gating", [False, True])
def test_n4_outputs_identical_with_and_without_planes(generic, gating, cuda, native_lib):
    """Position-only and generic dense-H updates, gated (displaced fixes) and not, full and packed covariances, both
    geodetic tiers, with and without a statistics tape, zero noise and noise tapes: every existing output bit-identical."""
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch

    tracks, dts = _fleet4(80, 40, seed=300 + 2 * generic + gating, k=2, outliers=0.05 if gating else 0.0)
    H, R = (H_DENSE, R_DENSE) if generic and not gating else (H_POS, R_GATE if gating else R_POS)
    for noise in ((None,) if gating else (None, _tapes4(tracks, dts, 5))):
        b = TrackBatch.from_tracks(tracks, dts, device=cuda, noise=noise)
        for packed in (False, True):
            for long_steps in (False, True):
                ukf = BatchedUKF(H, Q_DEF, R, P_DEF, gating=gating, force_generic=generic, packed_cov=packed, long_steps=long_steps)
                for reuse_stats in (True, False):
                    base = ukf.run(b, res=ukf.allocate(b, reuse_stats=reuse_stats)).to_host()
                    got = ukf.run(b, res=ukf.allocate(b, reuse_stats=reuse_stats, innovations=True)).to_host()
                    _assert_untouched(got)
                    for i in range(len(tracks)):
                        gi, bi = got.track(i), base.track(i)
                        assert "nis" in gi and "nis" not in bi
                        _same(gi, bi, KEYS4, (noise is not None, packed, long_steps, reuse_stats, i))
                    if gating:
                        assert int(base.gate_iters.sum()) > 0


@pytest.mark.parametrize("case", ["position", "dense", "gated", "gated_generic"])
@pytest.mark.parametrize("k", [1, 2])
def test_n4_statistics_against_numpy(case, k, cuda, native_lib):
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch

    gating = case.startswith("gated")
    generic = case in ("dense", "gated_generic")
    H, R = {"position": (H_POS, R_POS), "dense": (H_DENSE, R_DENSE), "gated": (H_POS, R_GATE), "gated_generic": (H_POS, R_GATE)}[case]
    tracks, dts = _fleet4(48, 36, seed=400 + k, k=k, outliers=0.05 if gating else 0.0)
    noise = None if gating else _tapes4(tracks, dts, 11 + k)
    ukf = BatchedUKF(H, Q_DEF, R, P_DEF, gating=gating, force_generic=generic)
    res = ukf.run(TrackBatch.from_tracks(tracks, dts, device=cuda, noise=noise), innovations=True)
    res.check_status()
    _assert_untouched(res)
    pos = not generic
    for i in range(len(tracks)):
        ref = _ref4(tracks[i], dts[i], tracks[i].z[:, 0], H, Q_DEF, R, P_DEF, gating=gating, noise=noise[i] if noise else None, pos=pos)
        _assert_stats(res.track(i), ref, (case, k, i))


def test_n4_statistics_follow_their_tracks(cuda, native_lib):
    """The planes follow their tracks through the length sort: any packing order gives the same track(i) statistics."""
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch

    tracks, dts = _fleet4(96, 30, seed=500, k=1, nobs_min=3)
    perm = np.random.default_rng(3).permutation(len(tracks))
    ukf = BatchedUKF(H_POS, Q_DEF, R_POS, P_DEF)
    a = ukf.run(TrackBatch.from_tracks(tracks, dts, device=cuda), innovations=True).to_host()
    b = ukf.run(TrackBatch.from_tracks([tracks[j] for j in perm], [dts[j] for j in perm], device=cuda, sort_by_length=False),
                innovations=True).to_host()
    for i, j in enumerate(perm):
        _same(b.track(i), a.track(int(j)), ("nis", "loglik", "innov_rank", "n_updates"), i)


def test_n4_run_many_and_partitioned(cuda, native_lib):
    """run_many with innovation planes equals run tile by tile, on the default and on the partitioned schedule; the
    fused pass refuses them."""
    import torch

    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.partition import SmPartition
    from ship_track_estimators_b200.synthetic import make_tracks

    ukf = BatchedUKF(H_POS, Q_DEF, R_GATE, P_DEF, gating=True, packed_cov=True)
    tiles = [TrackBatch.from_synthetic(make_tracks(1024, 60, seed=600 + i, device="cpu", outlier_frac=0.05, dts_choices=(1, 2, 3)),
                                       substeps=2, need_rows=ukf.model.rows_needed()).to(cuda) for i in range(3)]
    ref = [ukf.run(b, innovations=True) for b in tiles]
    names = ("mean_f", "cov_f", "mean_s", "cov_s", "status", "n_updates", "gate_iters", "nis", "loglik", "innov_rank")

    def same(rs):
        torch.cuda.synchronize()
        for r, g in zip(ref, rs):
            for name in names:
                assert torch.equal(getattr(r, name), getattr(g, name)) or name in ("nis", "loglik") and \
                    torch.equal(getattr(r, name).nan_to_num(7.0), getattr(g, name).nan_to_num(7.0)), name

    got = [ukf.allocate(b, innovations=True) for b in tiles]
    ukf.run_many(tiles, got)
    same(got)
    with SmPartition(cuda, smoother_sms=48) as part:
        got = [ukf.allocate(b, innovations=True) for b in tiles]
        ukf.run_many(tiles, got, partition=part)
        same(got)
    with pytest.raises(ValueError, match="innovation"):
        ukf.run_many(tiles, [ukf.allocate(b, innovations=True) for b in tiles], fused=True)


# --------------------------------------------------------------------------- #
# n = 5                                                                       #
# --------------------------------------------------------------------------- #
def _classes(T):
    """Two ship classes: GPS ships and historical logbook ships with their own Q and R."""
    from test_gpu_fleet_n5 import Q5, R5

    R_log, Q_log = R5.copy(), Q5 * 4.0
    R_log[0, 0] = R_log[1, 1] = 0.25
    R_log[0, 1] = R_log[1, 0] = 0.05
    return [Q5 if t % 2 == 0 else Q_log for t in range(T)], [R5 if t % 2 == 0 else R_log for t in range(T)]


def test_n5_outputs_identical_with_and_without_planes(cuda, native_lib):
    from test_gpu_fleet_n5 import H5, P5, Q5, R5, _fleet
    from test_gpu_fleet_n5_noise import _tapes

    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(96, 40, seed=700, nobs_min=4)
    T = len(tracks)
    Qs, Rs = _classes(T)
    engine = BatchedUKFN(H5, Q5, R5, P5)
    for noise in (None, _tapes(tracks, dts, 9)):
        for kw in (dict(), dict(Q=Qs, R=Rs), dict(R=Rs)):
            b = TrackBatchN.from_tracks(tracks, dts, x0=x0, noise=noise, device=cuda, **kw)
            base = engine.run(b).to_host()
            got = engine.run(b, innovations=True).to_host()
            _assert_untouched(got)
            for i in range(T):
                gi, bi = got.track(i), base.track(i)
                assert "loglik" in gi and "loglik" not in bi
                _same(gi, bi, ("means", "covs", "means_s", "covs_s", "status", "n_updates"), (noise is not None, sorted(kw), i))


@pytest.mark.parametrize("k", [1, 2])
def test_n5_statistics_against_numpy(k, cuda, native_lib):
    from test_gpu_fleet_n5 import H5, P5, Q5, R5, _fleet

    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(40, 30, seed=710 + k, ks=(k,), nobs_min=4)
    Qs, Rs = _classes(len(tracks))
    res = BatchedUKFN(H5, Q5, R5, P5).run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda, Q=Qs, R=Rs), innovations=True)
    res.check_status()
    _assert_untouched(res)
    for i in range(len(tracks)):
        ref = _ref5(tracks[i], dts[i], x0[i], H5, Qs[i], Rs[i], P5)
        _assert_stats(res.track(i), ref, (k, i))
        assert set(ref[:, 2]) == {4}   # R5 leaves the turn-rate row of S exactly zero: that eigenvalue is dropped


def test_n5_run_many_and_order(cuda, native_lib):
    import torch

    from test_gpu_fleet_n5 import H5, P5, Q5, R5, _fleet

    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(120, 30, seed=720, nobs_min=3)
    Qs, Rs = _classes(len(tracks))
    engine = BatchedUKFN(H5, Q5, R5, P5)
    tiles = TrackBatchN.fleet_tiles(tracks, dts, x0=x0, device=cuda, state_budget=1200, granule=8, Q=Qs, R=Rs)
    assert len(tiles) > 1
    ref = [engine.run(b, innovations=True) for b in tiles]
    got = [engine.allocate(b, innovations=True) for b in tiles]
    engine.run_many(tiles, got)
    torch.cuda.synchronize()
    one = engine.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda, Q=Qs, R=Rs), innovations=True).to_host()
    keys = ("means", "covs", "means_s", "covs_s", "status", "n_updates", "nis", "loglik", "innov_rank")
    for r, g in zip(ref, got):
        r, g = r.to_host(), g.to_host()
        for i in g.order:   # the caller's tracks this tile holds: run_many equals run, and both equal the one-tile run
            _same(g.track(int(i)), r.track(int(i)), keys, int(i))
            _same(g.track(int(i)), one.track(int(i)), ("nis", "loglik", "innov_rank"), int(i))


# --------------------------------------------------------------------------- #
# the use case: choosing R by maximum likelihood                             #
# --------------------------------------------------------------------------- #
SIGMA = 0.05                                 # degrees: the synthetic fixes' position noise (make_tracks' obs_sigma_deg)
SCALES = (0.25, 0.5, 1.0, 2.0, 4.0)          # candidate R / true position variance
# one fixed process noise for every candidate R (the synthetic ships' speed and course wander, with room for what the
# position-only filter does not model)
Q_ML4, P_ML4 = np.diag([1e-4, 1e-4, 0.2, 4.0]), np.diag([0.01, 0.01, 100.0, 900.0])
Q_ML5, P_ML5 = np.diag([1e-4, 1e-4, 0.2, 4.0, 1e-4]), np.diag([0.01, 0.01, 100.0, 900.0, 1e-2])


def _ml_fleet(T, seed):
    """Fixes with known position noise; the rate inputs are zero (make_tracks derives them from the noisy fixes, which
    would feed that noise into every predict as an unmodelled process noise)."""
    from ship_track_estimators_b200.synthetic import make_tracks

    syn = make_tracks(T, 80, seed=seed, device="cpu", obs_sigma_deg=SIGMA)
    tracks = []
    for t in range(T):
        z = np.stack([syn.lon[:, t].numpy(), syn.lat[:, t].numpy(), syn.sog[:, t].numpy(), syn.cog[:, t].numpy()])
        tracks.append(SimpleNamespace(dts=syn.dts[:, t].numpy().copy(), z=z, sog_rate=np.zeros(z.shape[1]), cog_rate=np.zeros(z.shape[1])))
    return tracks


def test_n5_maximum_likelihood_picks_the_true_r(cuda, native_lib):
    """One five-state tile holds the fleet five times, each copy with a candidate position R (per-track planes): the
    summed log-likelihood is largest at the true variance."""
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.performance_metrics import innovation_metrics

    fleet = _ml_fleet(256, seed=800)
    T = len(fleet)

    def R_of(s):
        return np.diag([s * SIGMA ** 2, s * SIGMA ** 2, 0.0, 0.0, 0.0])

    for tr in fleet:
        tr.z = np.vstack([tr.z, np.zeros((1, tr.z.shape[1]))])
    tracks = fleet * len(SCALES)
    b = TrackBatchN.from_tracks(tracks, [tr.dts for tr in tracks], x0=[tr.z[:, 0] for tr in tracks], device=cuda,
                                R=[R_of(s) for s in SCALES for _ in range(T)])
    res = BatchedUKFN(np.diag([1.0, 1.0, 0.0, 0.0, 0.0]), Q_ML5, R_of(1.0), P_ML5).run(b, smoother=False, innovations=True)
    res.check_status()
    m = innovation_metrics(res)
    assert m["loglik"].shape == (len(tracks),) and m["loglik"].device == res.nis.device
    cols = np.arange(len(tracks)) if b.order is None else np.asarray(b.order)   # tile column -> caller's index
    loglik, cand = m["loglik"].cpu().numpy(), cols // T
    total = np.array([loglik[cand == c].sum() for c in range(len(SCALES))])
    assert int(np.argmax(total)) == SCALES.index(1.0), total
    assert int(m["dof"].sum()) == 2 * int(m["n_updates"].sum())


def test_n4_maximum_likelihood_picks_the_true_r(cuda, native_lib):
    """The same selection on the four-state path: five BatchedUKF runs, one per candidate R."""
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.performance_metrics import innovation_metrics

    fleet = _ml_fleet(256, seed=810)
    b = TrackBatch.from_tracks(fleet, [tr.dts for tr in fleet], device=cuda)
    total = []
    for s in SCALES:
        res = BatchedUKF(H_POS, Q_ML4, np.diag([s * SIGMA ** 2, s * SIGMA ** 2, 0.0, 0.0]), P_ML4).run(b, smoother=False, innovations=True)
        res.check_status()
        m = innovation_metrics(res)
        total.append(float(m["loglik"].sum()))
        assert int(m["dof"].sum()) == 2 * int(m["n_updates"].sum())
    assert int(np.argmax(total)) == SCALES.index(1.0), total
