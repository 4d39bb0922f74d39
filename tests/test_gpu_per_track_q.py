"""GPU: per-track process noise on the n = 4 passes (``TrackBatch.Q``, ``ste_ukf_forward_noise_f64`` /
``ste_urtss_backward_noise_f64``) - planes that all hold the shared Q change no output bit, a tile of distinct per-track
matrices equals one-track runs with each track's Q as the filter's, two ship classes against the C oracle, the planes
following their tracks through the packing order and every schedule, and fit_noise(per="track") applied back to the
fleet."""
from types import SimpleNamespace

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

H_POS = np.diag([1.0, 1.0, 0.0, 0.0])
R_POS = np.diag([1e-3, 1e-3, 0.0, 0.0])
R_GATE = np.diag([0.05, 0.05, 0.0, 0.0])
Q_DEF = np.diag([1e-2, 1e-2, 1e-4, 1e-4])
P_DEF = np.eye(4)
H_DENSE = np.array([[1.0, 0.1, 0.0, 0.0], [0.05, 1.0, 0.0, 0.0], [0.0, 0.0, 1.0, 0.02], [0.0, 0.0, 0.01, 1.0]])
R_DENSE = np.array([[2e-3, 5e-4, 0.0, 0.0], [5e-4, 1e-3, 0.0, 0.0], [0.0, 0.0, 0.5, 0.1], [0.0, 0.0, 0.1, 4.0]])
RES = ("mean_f", "cov_f", "mean_s", "cov_s", "status", "n_updates", "gate_iters", "gate_lambda", "gate_scale", "smooth_stats",
       "nis", "loglik", "innov_rank")
KEYS = ("means", "covs", "means_s", "covs_s", "status", "n_updates", "gate_iters", "gate_lambda", "gate_scale", "nis", "loglik",
        "innov_rank")


@pytest.fixture(autouse=True, scope="module")
def _release_cached_blocks():
    yield
    import torch

    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _fleet(T, nobs_max, seed, k=1, outliers=0.0, nobs_min=5):
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


def _tapes(tracks, dts, seed):
    rng = np.random.default_rng(seed)
    return [dict(pred=rng.normal(size=(len(d), 4)), upd=rng.normal(size=(tr.z.shape[1], 4)), bwd=rng.normal(size=(len(d), 4)))
            for tr, d in zip(tracks, dts)]


def _track_qs(T, seed):
    """One positive-definite Q per track with correlated lon / lat and SOG / COG entries."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(T):
        v = np.array([1e-2, 1e-2, 1e-4, 1e-4]) * rng.uniform(0.2, 5.0, size=4)
        rho_pos, rho_vel = rng.uniform(-0.8, 0.8, size=2)
        Q = np.diag(v)
        Q[0, 1] = Q[1, 0] = rho_pos * np.sqrt(v[0] * v[1])
        Q[2, 3] = Q[3, 2] = rho_vel * np.sqrt(v[2] * v[3])
        out.append(Q)
    return out


def _same_results(a, b, where):
    import torch

    for name in RES:
        x, y = getattr(a, name), getattr(b, name)
        assert (x is None) == (y is None), (where, name)
        if x is not None:
            if x.dtype == torch.float64:
                x, y = x.nan_to_num(7.0), y.nan_to_num(7.0)   # NaN rows (innovation planes past n_updates) compare equal
            assert torch.equal(x, y), (where, name)


def _alloc(ukf, b, **kw):
    """Result buffers whose rows past a ragged track's end (never written) hold zeros, so whole tensors compare."""
    res = ukf.allocate(b, **kw)
    for name in ("mean_f", "cov_f", "mean_s", "cov_s", "smooth_stats"):
        if getattr(res, name) is not None:
            getattr(res, name).zero_()
    return res


def _written(t, n_steps):
    """The states [S][planes][T] a pass writes: rows 0 .. n_steps[t] of column t (the others zeroed)."""
    import torch

    rows = torch.arange(t.shape[0], device=t.device)[:, None] <= n_steps.to(t.device)[None, :]
    return torch.where(rows[:, None, :], t, torch.zeros((), dtype=t.dtype, device=t.device))


def _same_tracks(a, b, keys, where):
    for key in keys:
        assert (key in a) == (key in b), (where, key)
        if key in a:
            assert np.array_equal(a[key], b[key]), (where, key)


@pytest.mark.parametrize("case", ["position", "dense", "gated"])
@pytest.mark.parametrize("k", [1, 2])
def test_planes_holding_the_shared_q_change_nothing(case, k, cuda, native_lib):
    """Per-track planes that all hold the filter's Q: every output - states, covariances (packed and full), smoothed states,
    status, n_updates, gating planes, innovation planes, the smoother tape - bit-identical to the tile without planes, with
    and without the tape, with zero noise and noise tapes."""
    import torch

    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch

    gating = case == "gated"
    H, R = {"position": (H_POS, R_POS), "dense": (H_DENSE, R_DENSE), "gated": (H_POS, R_GATE)}[case]
    tracks, dts = _fleet(72, 30, seed=800 + 10 * k + len(case), k=k, outliers=0.05 if gating else 0.0)
    for noise in ((None,) if gating else (None, _tapes(tracks, dts, 3 + k))):
        b = TrackBatch.from_tracks(tracks, dts, device=cuda, noise=noise)
        qb = b.with_noise(Q=[Q_DEF] * len(tracks))
        for packed in (False, True):
            ukf = BatchedUKF(H, Q_DEF, R, P_DEF, gating=gating, force_generic=case == "dense", packed_cov=packed)
            for reuse_stats in (True, False):
                for innovations in (False, True):
                    base = ukf.run(b, res=_alloc(ukf, b, reuse_stats=reuse_stats, innovations=innovations))
                    got = ukf.run(qb, res=_alloc(ukf, qb, reuse_stats=reuse_stats, innovations=innovations))
                    torch.cuda.synchronize()
                    _same_results(base, got, (noise is not None, packed, reuse_stats, innovations))
                    if gating:
                        assert int(base.gate_iters.sum()) > 0


@pytest.mark.parametrize("case", ["tape", "no_tape", "noise_tapes", "gated", "per_track_r"])
def test_distinct_q_equals_one_track_runs(case, cuda, native_lib):
    """A ragged tile where every track has its own Q (correlated lon / lat and SOG / COG entries): each track bit-identical
    to a one-track run of a filter built with that Q.  long_steps is pinned on both sides (the geodetic tier is chosen per
    tile, and the two tiers agree only to 1 ulp)."""
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch

    gating = case == "gated"
    tracks, dts = _fleet(70, 36, seed=900 + len(case), k=2 if case == "no_tape" else 1, outliers=0.05 if gating else 0.0, nobs_min=3)
    T = len(tracks)
    Qs = _track_qs(T, 17)
    noise = _tapes(tracks, dts, 21) if case == "noise_tapes" else None
    R = R_GATE if gating else R_POS
    Rs = None
    if case == "per_track_r":
        rng = np.random.default_rng(5)
        Rs = [np.diag([1e-3, 1e-3, 0.5, 4.0]) * rng.uniform(0.5, 2.0) for _ in range(T)]
    reuse_stats = case != "no_tape"
    for long_steps in (False, True):
        ukf = BatchedUKF(H_POS, Q_DEF, R, P_DEF, gating=gating, long_steps=long_steps)
        b = TrackBatch.from_tracks(tracks, dts, device=cuda, noise=noise, Q=Qs, R=Rs)
        res = ukf.run(b, res=ukf.allocate(b, reuse_stats=reuse_stats, innovations=True)).to_host()
        for i in range(T):
            one = BatchedUKF(H_POS, Qs[i], R, P_DEF, gating=gating, long_steps=long_steps)
            ob = TrackBatch.from_tracks([tracks[i]], [dts[i]], device=cuda, noise=None if noise is None else [noise[i]],
                                        R=None if Rs is None else [Rs[i]])
            ref = one.run(ob, res=one.allocate(ob, reuse_stats=reuse_stats, innovations=True)).to_host()
            _same_tracks(res.track(i), ref.track(0), KEYS, (case, long_steps, i))


def test_two_ship_classes_against_the_c_oracle(cuda, native_lib):
    """GPS ships and logbook ships with their own Q (every track carries its class's matrix) against the plain-C oracle run
    with that Q, filtered and smoothed, at 1e-9."""
    from _helpers import assert_track_close

    from oracle import ukf_c as OC
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch

    tracks, dts = _fleet(96, 40, seed=950, k=2, nobs_min=4)
    q_gps = Q_DEF
    q_log = np.array([[4e-2, 1e-2, 0.0, 0.0], [1e-2, 3e-2, 0.0, 0.0], [0.0, 0.0, 1e-3, 2e-4], [0.0, 0.0, 2e-4, 4e-3]])
    Qs = [q_gps if t % 2 == 0 else q_log for t in range(len(tracks))]
    res = BatchedUKF(H_POS, Q_DEF, R_POS, P_DEF).run(TrackBatch.from_tracks(tracks, dts, device=cuda, Q=Qs)).to_host()
    res.check_status()
    for i, tr in enumerate(tracks):
        ref = OC.run_track(tr.z[:, 0], P_DEF, H_POS, Qs[i], R_POS, dts[i], tr.dts, tr.z, tr.sog_rate, tr.cog_rate)
        assert_track_close(res.track(i), ref, label=f"per_track_q_classes[{i}]")


def test_order_and_schedules(cuda, native_lib):
    """Any packing order gives the same track(i); run_many, the partitioned schedule and run_host_pipelined equal run bit
    for bit."""
    import torch

    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.partition import SmPartition

    tracks, dts = _fleet(300, 40, seed=970, nobs_min=3)
    T = len(tracks)
    Qs = _track_qs(T, 29)
    ukf = BatchedUKF(H_POS, Q_DEF, R_POS, P_DEF, packed_cov=True, long_steps=False)
    a = ukf.run(TrackBatch.from_tracks(tracks, dts, device=cuda, Q=Qs)).to_host()
    perm = np.random.default_rng(3).permutation(T)
    b = ukf.run(TrackBatch.from_tracks([tracks[j] for j in perm], [dts[j] for j in perm], device=cuda, Q=[Qs[j] for j in perm],
                                       sort_by_length=False)).to_host()
    for i, j in enumerate(perm):
        _same_tracks(b.track(i), a.track(int(j)), ("means", "covs", "means_s", "covs_s", "status", "n_updates"), i)

    # equal-shape tiles (the host pipeline needs one shape), each with its own per-track Q
    parts = [np.arange(s, s + 100) for s in (0, 100, 200)]
    tiles = [TrackBatch.from_tracks([tracks[j] for j in p], [dts[j] for j in p], device="cpu", Q=[Qs[j] for j in p],
                                    sort_by_length=False) for p in parts]
    N = max(t.max_steps for t in tiles)
    M = max(t.max_obs for t in tiles)
    tiles = [_pad(t, N, M) for t in tiles]
    dev_tiles = [t.to(cuda) for t in tiles]
    ref = [ukf.run(t) for t in dev_tiles]
    torch.cuda.synchronize()
    names = ("mean_f", "cov_f", "mean_s", "cov_s", "status", "n_updates")

    def same(rs):
        torch.cuda.synchronize()
        for t, r, g in zip(tiles, ref, rs):
            for name in names:
                x, y = getattr(r, name), getattr(g, name)
                if x.dim() == 3:
                    x, y = _written(x, t.n_steps), _written(y, t.n_steps)
                assert torch.equal(x.cpu(), y.cpu()), name

    got = [ukf.allocate(t) for t in dev_tiles]
    ukf.run_many(dev_tiles, got)
    same(got)
    with SmPartition(cuda, smoother_sms=48) as part:
        got = [ukf.allocate(t) for t in dev_tiles]
        ukf.run_many(dev_tiles, got, partition=part)
        same(got)
    with pytest.raises(ValueError, match="per-track Q"):
        ukf.run_many(dev_tiles, [ukf.allocate(t) for t in dev_tiles], fused=True)
    pinned = [t.pin_memory() for t in tiles]
    assert all(p.Q is not None and p.Q.is_pinned() for p in pinned)
    outs = [ukf.host_outputs(pinned[0], outputs="all") for _ in pinned]
    moved = ukf.run_host_pipelined(pinned, outs, device=cuda, outputs="all")
    torch.cuda.synchronize()
    assert moved["h2d_bytes"] == sum(p.input_bytes() for p in pinned)
    same([SimpleNamespace(**o) for o in outs])


def _pad(b, N, M):
    """The tile with max_steps N and max_obs M (zero rows past each track's end, which no kernel reads)."""
    import torch

    from ship_track_estimators_b200.batch import TrackBatch

    def grow(t, rows):
        if t is None or t.shape[0] == rows:
            return t
        out = torch.zeros((rows,) + tuple(t.shape[1:]), dtype=t.dtype)
        out[: t.shape[0]] = t
        return out

    kw = {n: getattr(b, n) for n in TrackBatch._TENSORS}
    for n in ("dt", "upd_mask"):
        kw[n] = grow(kw[n], N)
    for n in ("sog_rate", "cog_rate"):
        kw[n] = grow(kw[n], M)
    return TrackBatch(z=[grow(r, M) for r in b.z], substeps=b.substeps, rate_repeat_all=b.rate_repeat_all,
                      n_steps_host=b.n_steps_host, order=b.order, **kw)


def test_fit_noise_per_track_then_apply(cuda, native_lib):
    """fit_noise(per="track") over a grid of Q scales, then from_tracks(Q=fit["Q"]) run with innovation planes: each
    track's log-likelihood, summed in update order, equals its chosen score bit for bit."""
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.tuning import fit_noise, noise_grid

    tracks, dts = _fleet(160, 40, seed=990, nobs_min=4)
    ukf = BatchedUKF(H_POS, Q_DEF, R_POS, P_DEF, long_steps=False)
    grid = noise_grid(Q_DEF, R_POS, q_scales=(0.1, 0.3, 1.0, 3.0, 10.0), r_scales=(1.0,))
    fit = fit_noise(ukf, TrackBatch.from_tracks(tracks, dts, device=cuda), grid, per="track")
    assert len(set(fit["best"].tolist())) > 1   # the tracks do not all choose the same Q
    res = ukf.run(TrackBatch.from_tracks(tracks, dts, device=cuda, Q=fit["Q"]), smoother=False, innovations=True).to_host()
    for i in range(len(tracks)):
        total = 0.0
        for v in res.track(i)["loglik"]:
            total += float(v)
        assert total == fit["loglik"][fit["best"][i], i], i
    # the same through with_noise on a tile built without matrices
    b = TrackBatch.from_tracks(tracks, dts, device=cuda)
    res2 = ukf.run(b.with_noise(Q=fit["Q"]), smoother=False, innovations=True).to_host()
    for i in range(len(tracks)):
        _same_tracks(res2.track(i), res.track(i), ("means", "covs", "loglik", "nis", "innov_rank"), i)
