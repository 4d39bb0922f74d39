"""GPU: per-track process and measurement noise on the five-state fleet path (``TrackBatchN.Q`` / ``R``, ``SteNoiseN``
through ``ste_ukf_forward_noise_n_f64`` / ``ste_urtss_backward_tracks_noise_n_f64``) - the shared path unchanged, every
track bit-identical to a filter built with its own matrices, the numpy oracle for a fleet of two ship classes, tiling, the
host pipeline, track order, device ingest and estimate_fleet's ship_settings."""
import os
from types import SimpleNamespace

import numpy as np
import pytest

from _helpers import TOL
from test_gpu_fleet_n5 import H5, P5, Q5, R5, _errs, _fleet

pytestmark = pytest.mark.gpu

KEYS = ("means", "covs", "means_s", "covs_s", "status", "n_updates")


@pytest.fixture(autouse=True, scope="module")
def _release_cached_blocks():
    yield
    import torch

    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _noise(T, seed):
    """Distinct symmetric Q and R per track: the shared diagonals scaled per track, with lon / lat and SOG / COG
    correlations (every off-diagonal plane the kernels read is exercised)."""
    rng = np.random.default_rng(seed)
    Qs, Rs = [], []
    for _ in range(T):
        q = np.diag(Q5).copy() * rng.uniform(0.3, 3.0, 5)
        r = np.diag(R5).copy() * rng.uniform(0.3, 3.0, 5)
        r[4] = rng.choice([0.0, 1e-2])
        Q, R = np.diag(q), np.diag(r)
        for M, v in ((Q, q), (R, r)):
            for i, j in ((0, 1), (2, 3)):
                M[i, j] = M[j, i] = rng.uniform(-0.4, 0.4) * np.sqrt(v[i] * v[j])
        Qs.append(Q)
        Rs.append(R)
    return Qs, Rs


def _tapes(tracks, dts, seed):
    rng = np.random.default_rng(seed)
    return [dict(pred=rng.normal(size=(len(d), 5)), upd=rng.normal(size=(tr.z.shape[1], 5)), bwd=rng.normal(size=(len(d), 5)))
            for tr, d in zip(tracks, dts)]


def _same(a, b, where):
    for key in KEYS:
        if key in a:
            assert np.array_equal(a[key], b[key]), (where, key)


def test_shared_matrices_as_planes_change_nothing(cuda, native_lib):
    """Planes that all hold the filter's Q / R (both, or one of them) give bit-identical forward and backward results,
    with zero noise and with tapes."""
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(96, 60, seed=101, nobs_min=5)
    T = len(tracks)
    engine = BatchedUKFN(H5, Q5, R5, P5)
    for noise in (None, _tapes(tracks, dts, 7)):
        base = engine.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, noise=noise, device=cuda)).to_host()
        for kw in (dict(Q=[Q5] * T, R=[R5] * T), dict(Q=[Q5] * T), dict(R=[R5] * T)):
            got = engine.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, noise=noise, device=cuda, **kw)).to_host()
            for i in range(T):
                _same(got.track(i), base.track(i), (noise is not None, sorted(kw), i))


def test_each_track_equals_a_filter_with_its_own_matrices(cuda, native_lib):
    """A ragged tile of 64 tracks with distinct Q and R: every track bit-identical to a one-track BatchedUKFN(H, Q_t, R_t, P)
    run (means, covariances, smoothed states, status), with zero noise and with tapes scaled by each track's diagonals."""
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(64, 67, seed=111, nobs_min=6)
    lens = [len(d) for d in dts]
    assert min(lens) >= 5 and max(lens) >= 100
    Qs, Rs = _noise(64, 3)
    engine = BatchedUKFN(H5, Q5, R5, P5)
    for noise in (None, _tapes(tracks, dts, 9)):
        res = engine.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, noise=noise, device=cuda, Q=Qs, R=Rs)).to_host()
        for i in range(64):
            one = BatchedUKFN(H5, Qs[i], Rs[i], P5).run(
                TrackBatchN.from_tracks([tracks[i]], [dts[i]], x0=[x0[i]], noise=None if noise is None else [noise[i]], device=cuda))
            got = res.track(i)
            assert np.count_nonzero(got["covs"][-1]) == 25
            _same(got, one.track(0), (noise is not None, i))


def test_two_ship_classes_against_the_numpy_oracle(cuda, native_lib):
    """256 ragged tracks, half logbook ships (R = 0.25 deg^2 on the position, a small turn-rate Q) and half GPS ships
    (R = 1e-3, a larger turn-rate Q), in one tile: each track against the n = 5 oracle with its own matrices at 1e-9."""
    import _oracle_n5 as O5
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(256, 151, seed=131, ks=(1, 2), nobs_min=20)
    classes = {"logbook": (np.diag([1e-2, 1e-2, 1e-4, 1e-4, 1e-6]), np.diag([0.25, 0.25, 0.5, 4.0, 0.0])),
               "gps": (np.diag([1e-2, 1e-2, 1e-4, 1e-4, 1e-4]), np.diag([1e-3, 1e-3, 0.5, 4.0, 0.0]))}
    kind = ["logbook" if i % 2 else "gps" for i in range(256)]
    Qs, Rs = [classes[k][0] for k in kind], [classes[k][1] for k in kind]
    res = BatchedUKFN(H5, Q5, R5, P5).run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda, Q=Qs, R=Rs)).to_host()
    res.check_status()
    worst = {k: np.zeros(4) for k in classes}
    for i, (tr, dt) in enumerate(zip(tracks, dts)):
        ref = O5.run_track(x0[i], P5, H5, Qs[i], Rs[i], dt, tr.dts, tr.z, tr.sog_rate)
        got = res.track(i)
        e = _errs(got["means"], got["covs"], ref["means"], ref["covs"]) + _errs(got["means_s"], got["covs_s"], ref["means_s"], ref["covs_s"])
        worst[kind[i]] = np.fmax(worst[kind[i]], e)
        assert max(e) <= TOL, (i, kind[i], e)
    for k, w in worst.items():
        print(f"  n = 5 per-track noise, {k} ships vs numpy oracle, worst (filtered mean, cov, smoothed mean, cov): {w}")


def test_tiles_pipeline_and_track_order(cuda, native_lib):
    """fleet_tiles + run_many equal one tile; a shuffled caller order leaves every track bit-identical (the matrices follow
    their tracks through the length sort); run_host_pipelined "cli" / "summary" equal run + the copy-out."""
    import torch

    from ship_track_estimators_b200.batch import TrackBatch
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.performance_metrics import track_metrics
    from ship_track_estimators_b200.synthetic import make_tracks

    tracks, dts, x0 = _fleet(2000, 60, seed=141, ks=(1, 2), nobs_min=3)
    Qs, Rs = _noise(2000, 5)
    ukf = BatchedUKFN(H5, Q5, R5, P5)
    whole = ukf.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda, Q=Qs, R=Rs)).to_host()
    tiles = TrackBatchN.fleet_tiles(tracks, dts, x0=x0, device=cuda, state_budget=40_000, granule=128, Q=Qs, R=Rs)
    assert len(tiles) >= 3
    results = [ukf.allocate(t) for t in tiles]
    ukf.run_many(tiles, results)
    seen = 0
    for tile, res in zip(tiles, results):
        host = res.to_host()
        for i in tile.order:
            _same(host.track(int(i)), whole.track(int(i)), ("tiles", int(i)))
            seen += 1
    assert seen == len(tracks)
    del results, tiles

    perm = np.random.default_rng(2).permutation(len(tracks))
    pick = lambda seq: [seq[j] for j in perm]   # noqa: E731
    shuffled = ukf.run(TrackBatchN.from_tracks(pick(tracks), pick(dts), x0=pick(x0), device=cuda, Q=pick(Qs), R=pick(Rs))).to_host()
    for k, j in enumerate(perm):
        _same(shuffled.track(k), whole.track(int(j)), ("shuffled", k))

    dev_tiles = []
    for j in range(3):
        syn = make_tracks(256, 41, seed=150 + j, device="cuda", dts_choices=(1.0, 2.0), nobs_min=20)
        q, r = _noise(256, 160 + j)
        dev_tiles.append(TrackBatchN.from_batch(TrackBatch.from_synthetic(syn, substeps=2, need_rows=(True,) * 4), turn_rate0=0.05, Q=q, R=r))
    full = [ukf.run(t) for t in dev_tiles]
    pinned = [t.pin_memory() for t in dev_tiles]
    assert pinned[0].Q.is_pinned() and pinned[0].R.is_pinned()
    diag = [0, 6, 12, 18, 24]
    for name in ("cli", "summary"):
        outs = [ukf.host_outputs(pinned[0], outputs=name) for _ in pinned]
        ukf.run_host_pipelined(pinned, outs, device=cuda, outputs=name)
        torch.cuda.synchronize()
        for o, f, t in zip(outs, full, dev_tiles):
            assert torch.equal(o["status"], f.status.cpu()) and torch.equal(o["n_updates"], f.n_updates.cpu())
            nsteps = torch.from_numpy(t.n_steps_host.astype(np.int64))
            valid = (torch.arange(f.mean_f.shape[0])[:, None, None] <= nsteps[None, None, :]).double()
            for key in ukf.OUTPUT_SETS[name]:
                if key in ("mean_f", "mean_s"):
                    want = getattr(f, key).cpu()
                elif key.startswith("diag"):
                    want = (f.cov_f if key == "diag_f" else f.cov_s)[:, diag, :].cpu()
                elif key == "final":
                    cols = torch.arange(len(nsteps))
                    want = torch.cat([f.mean_f.cpu()[nsteps, :, cols].T, f.cov_f.cpu()[nsteps, :, cols].T], dim=0)
                else:
                    m = track_metrics(ukf, t, f, which="smoothed")
                    want = torch.cat([m["rmse"], m["cum_abs"], m["max_abs"]], dim=0).cpu()
                w = valid if want.dim() == 3 else 1.0
                assert torch.equal(torch.nan_to_num(o[key]) * w, torch.nan_to_num(want) * w), (name, key)


def test_device_ingest_gets_each_ships_matrices(cuda, native_lib, tmp_path):
    """A CSV read by the device reader and by the host reader, through the same from_batch(..., Q=, R=): bit-identical per
    ship, and each ship equal to its column of the tile run with that ship's matrices as the filter's shared ones."""
    from test_host_dropin import _fleet_csv

    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.ingest import read_csv_fleet, read_csv_fleet_device

    csv = str(tmp_path / "fleet.csv")
    _fleet_csv(csv, seed=21, n_ships=24, string_labels=False, time_ordered=True)
    host_all = read_csv_fleet(csv, id_col="primary.id")
    ids = [s for s, m in zip(host_all.ids, host_all.n_obs) if m >= 3]
    assert len(ids) >= 12
    Qs, Rs = _noise(len(ids), 17)
    fh = read_csv_fleet(csv, id_col="primary.id", ship_ids=ids)
    fd = read_csv_fleet_device(csv, id_col="primary.id", ship_ids=ids, device=cuda)
    assert list(fh.ids) == list(fd.ids) == ids
    bh, bd = fh.to_batch(device=cuda, substeps=2), fd.to_batch(substeps=2)
    assert bd.order is not None and list(bd.order) != list(range(len(ids)))
    engine = BatchedUKFN(H5, Q5, R5, P5)
    rh = engine.run(TrackBatchN.from_batch(bh, turn_rate0=0.1, Q=Qs, R=Rs)).to_host()
    rd = engine.run(TrackBatchN.from_batch(bd, turn_rate0=0.1, Q=Qs, R=Rs)).to_host()
    for i in range(len(ids)):
        _same(rd.track(i), rh.track(i), ("host reader", ids[i]))
        own = BatchedUKFN(H5, Qs[i], Rs[i], P5).run(TrackBatchN.from_batch(bd, turn_rate0=0.1)).to_host()
        _same(rd.track(i), own.track(i), ("own matrices", ids[i]))


@pytest.mark.parametrize("formatter", ["host", "device"])
def test_estimate_fleet_ship_settings_files(formatter, cuda, native_lib, tmp_path):
    """estimate_fleet at dim 5 with ship_settings for some ships, on one tile and on several: every overridden ship's files
    byte-identical to write_track_outputs of the class API run with its Q / R, every other ship's to a run without
    ship_settings."""
    from test_host_dropin import _fleet_csv

    from ship_track_estimators_b200.cli.main_cli import _get_input_matrix
    from ship_track_estimators_b200.cli.writers import estimate_fleet, write_track_outputs
    from ship_track_estimators_b200.kalman_filters import UnscentedKalmanFilter, geodetic_dynamics_turn
    from ship_track_estimators_b200.utils import generate_dts

    csv = str(tmp_path / "fleet.csv")
    _fleet_csv(csv, seed=35, n_ships=30, time_ordered=True)
    settings = {"dim": 5, "H": [1, 1, 0, 0, 0], "R": [0.001, 0.001, 0, 0, 0], "Q": [1e-2, 1e-2, 1e-4, 1e-4, 1e-5],
                "P": [1.0, 1.0, 1.0, 4.0, 1e-2], "dt": -1, "nsteps": 2, "smooth": 2}
    kw = dict(id_col="primary.id", lat_col="lat", lon_col="lon", apply_rts_smoother=True, device=cuda, formatter=formatter)
    plain = str(tmp_path / "plain")
    os.makedirs(plain)
    fleet, _ = estimate_fleet(csv, settings, directory=plain, **kw)
    ids = list(fleet.ids)
    gps = [[1e-3, 1e-4, 0, 0, 0], [1e-4, 1e-3, 0, 0, 0], [0, 0, 0, 0, 0], [0, 0, 0, 0, 0], [0, 0, 0, 0, 0]]
    ship_settings = {ids[1]: {"R": [0.25, 0.25, 0, 0, 0]}, ids[4]: {"Q": [1e-2, 1e-2, 1e-4, 1e-4, 1e-3], "R": gps},
                     ids[-1]: {"Q": [2e-2, 2e-2, 1e-4, 1e-4, 1e-6]}}
    one, tiled, ref = (str(tmp_path / d) for d in ("one", "tiled", "ref"))
    for d in (one, tiled, ref):
        os.makedirs(d)
    f1, res = estimate_fleet(csv, settings, directory=one, ship_settings=ship_settings, **kw)
    ft, res_t = estimate_fleet(csv, settings, directory=tiled, ship_settings=ship_settings,
                               tile_plan=dict(state_budget=300, granule=4), **kw)
    assert res is not None and res_t is None and list(f1.ids) == list(ft.ids) == ids

    H, Q, R, P = (_get_input_matrix(settings, k, 5) for k in ("H", "Q", "R", "P"))
    b4 = fleet.to_batch(device=cuda, substeps=2, smooth_width=2, need_rows=(True,) * 4, geodesy="wgs84")
    col_of = np.arange(fleet.n_tracks) if b4.order is None else np.argsort(b4.order)
    rows = [r.cpu().numpy() for r in b4.z]
    sr, cr = b4.sog_rate.cpu().numpy(), b4.cog_rate.cpu().numpy()
    for sid, over in ship_settings.items():
        i = ids.index(sid)
        lat, lon, dts = fleet.track(i)
        j, m = int(col_of[i]), int(fleet.n_obs[i])
        st = SimpleNamespace(dts=dts, z=np.stack([r[:m, j] for r in rows]), sog_rate=sr[:m, j], cog_rate=cr[:m, j])
        dt = generate_dts(dts, 2)
        Qi = _get_input_matrix(over, "Q", 5) if "Q" in over else Q
        Ri = _get_input_matrix(over, "R", 5) if "R" in over else R
        ukf = UnscentedKalmanFilter(H=H, Q=Qi, R=Ri, P=P, x0=np.append(st.z[:, 0], 0.0), non_linear_process=geodetic_dynamics_turn,
                                    noise="zero")
        means, covs = ukf.run(len(dt), dt, st)
        means_s, covs_s = ukf.run_rts_smoother(st)
        write_track_outputs("output", sid, means, covs, dt, lon, lat, means_s, covs_s, ref)
    names = sorted(os.listdir(plain))
    assert len(names) == 6 * len(ids) and sorted(os.listdir(one)) == names and sorted(os.listdir(tiled)) == names
    overridden = set(os.listdir(ref))
    assert len(overridden) == 6 * len(ship_settings)
    changed = 0
    for name in names:
        want = open(os.path.join(ref if name in overridden else plain, name), "rb").read()
        assert open(os.path.join(one, name), "rb").read() == want, name
        assert open(os.path.join(tiled, name), "rb").read() == want, name
        changed += name in overridden and "predictions" in name and want != open(os.path.join(plain, name), "rb").read()
    assert changed == 2 * len(ship_settings)   # the overrides changed every overridden ship's states
