"""GPU: the five-state fleet path at scale - fit metrics on the device (``ste_track_metrics_n_f64``), ragged tiling with
``run_many``, the pinned-host pipeline per output set, ``estimate_fleet`` at ``dim: 5`` and ``sharding.local_summary``."""
import os
from types import SimpleNamespace

import numpy as np
import pytest

from test_gpu_fleet_n5 import H5, P5, Q5, R5, _fleet

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, scope="module")
def _release_cached_blocks():
    yield
    import torch

    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _synthetic_tile(seed, T=256, nobs=41, k=2):
    """A ragged five-state device tile of fixed shape (max_steps = (nobs - 1) k whatever the lengths)."""
    from ship_track_estimators_b200.batch import TrackBatch
    from ship_track_estimators_b200.batch_n import TrackBatchN
    from ship_track_estimators_b200.synthetic import make_tracks

    syn = make_tracks(T, nobs, seed=seed, device="cuda", dts_choices=(1.0, 2.0), nobs_min=20)
    return TrackBatchN.from_batch(TrackBatch.from_synthetic(syn, substeps=k, need_rows=(True,) * 4), turn_rate0=0.05)


@pytest.mark.parametrize("k,rows", [(1, 5), (2, 4)])
def test_track_metrics_n5_against_the_oracle(k, rows, cuda, native_lib):
    """Per-track rmse / cum_abs / max_abs / abs_diff of the filtered and the smoothed states of a ragged tile against the
    oracle's restatement of performance_metrics.py on the same states; NaN rows and pair counts exact."""
    import torch

    from oracle import ukf_numpy as O
    from ship_track_estimators_b200.batch import exact_update_mask
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.performance_metrics import track_metrics

    tracks, dts, x0 = _fleet(160, 50, seed=60 + k, ks=(k,), nobs_min=5)
    if rows == 4:
        for tr in tracks:
            tr.z = tr.z[:4]
    b = TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda)
    if rows == 4:
        b.z[4] = None
    ukf = BatchedUKFN(H5, Q5, R5, P5)
    res = ukf.run(b)
    host = res.to_host()
    for which, key in (("filtered", "means"), ("smoothed", "means_s")):
        got = {n: v.cpu().numpy() for n, v in track_metrics(ukf, b, res, which=which, keep_abs_diff=True).items()}
        assert got["rmse"].shape == (5, len(tracks)) and got["abs_diff"].shape == (b.max_obs, 5, len(tracks))
        for r in range(rows, 5):
            assert np.isnan(got["rmse"][r]).all() and np.isnan(got["abs_diff"][:, r]).all()
        for i, tr in enumerate(tracks):
            j = host.column(i)
            z = np.zeros((5, tr.z.shape[1]))
            z[: tr.z.shape[0]] = tr.z
            ref = O.track_metrics(host.track(i)[key], exact_update_mask(dts[i], tr.dts), z, rows=range(rows))
            n = len(ref[0]["abs_diff"])
            assert int(got["n_pairs"][j]) == n, (which, i)
            for r in range(rows):
                assert np.array_equal(got["abs_diff"][:n, r, j], ref[r]["abs_diff"]), (which, i, r)
                assert np.isnan(got["abs_diff"][n:, r, j]).all()
                assert got["max_abs"][r, j] == ref[r]["max_abs"]
                np.testing.assert_allclose(got["cum_abs"][r, j], ref[r]["cum_abs"], rtol=1e-12)
                np.testing.assert_allclose(got["rmse"][r, j], ref[r]["rmse"], rtol=1e-12)
    del res
    torch.cuda.empty_cache()


def test_n4_metrics_equal_the_n5_kernel_on_the_same_states(cuda, native_lib):
    """ste_track_metrics_f64 on an n = 4 tile and ste_track_metrics_n_f64 on its five-state form (from_batch) fed the same
    means (padded with a fifth row) give bit-identical rows 0-3: the two instantiations share their arithmetic."""
    import torch

    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN, TrackResultsN
    from ship_track_estimators_b200.performance_metrics import track_metrics
    from ship_track_estimators_b200.synthetic import make_tracks

    syn = make_tracks(300, 70, seed=93, device="cpu", dts_choices=(1, 2, 3), nobs_min=5)
    H4, R4 = np.diag([1.0, 1, 1, 1]), np.diag([1e-3, 1e-3, 0.5, 4.0])
    u4 = BatchedUKF(H4, Q5[:4, :4], R4, P5[:4, :4])
    b4 = TrackBatch.from_synthetic(syn, substeps=2, need_rows=u4.model.rows_needed()).to(cuda)
    r4 = u4.run(b4)
    b5 = TrackBatchN.from_batch(b4)
    u5 = BatchedUKFN(np.pad(H4, ((0, 1), (0, 1))), Q5, np.pad(R4, ((0, 1), (0, 1))), P5)
    pad = lambda m: torch.cat([m, torch.zeros_like(m[:, :1])], dim=1).contiguous()   # noqa: E731
    S, T = r4.mean_f.shape[0], b4.n_tracks
    r5 = TrackResultsN(mean_f=pad(r4.mean_f), cov_f=torch.zeros(S, 25, T, dtype=torch.float64, device=cuda), mean_s=pad(r4.mean_s),
                       cov_s=torch.zeros(S, 25, T, dtype=torch.float64, device=cuda), status=r4.status, n_updates=r4.n_updates)
    for which in ("filtered", "smoothed"):
        m4 = track_metrics(u4, b4, r4, which=which, keep_abs_diff=True)
        m5 = track_metrics(u5, b5, r5, which=which, keep_abs_diff=True)
        assert torch.equal(m4["n_pairs"], m5["n_pairs"])
        for key in ("rmse", "cum_abs", "max_abs"):
            assert torch.equal(m4[key], m5[key][:4]) and bool(torch.isnan(m5[key][4]).all()), (which, key)
        assert torch.equal(torch.nan_to_num(m4["abs_diff"], nan=-1.0), torch.nan_to_num(m5["abs_diff"][:, :4], nan=-1.0))


def test_fleet_tiles_run_many_equal_one_tile(cuda, native_lib):
    """~3 000 ragged tracks cut into several tiles and run with run_many: every track bit-identical to one tile holding
    the whole fleet, looked up by the caller's index."""
    import torch

    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(3000, 60, seed=71, ks=(1, 2), nobs_min=3)
    ukf = BatchedUKFN(H5, Q5, R5, P5)
    tiles = TrackBatchN.fleet_tiles(tracks, dts, x0=x0, device=cuda, state_budget=60_000, granule=128)
    assert len(tiles) >= 3 and sum(t.n_tracks for t in tiles) == len(tracks)
    results = [ukf.allocate(t) for t in tiles]
    ukf.run_many(tiles, results)
    whole = ukf.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda)).to_host()
    seen = 0
    for tile, res in zip(tiles, results):
        host = res.to_host()
        for i in tile.order:
            a, b = host.track(int(i)), whole.track(int(i))
            for key in ("means", "covs", "means_s", "covs_s", "status", "n_updates"):
                assert np.array_equal(a[key], b[key]), (int(i), key)
            seen += 1
    assert seen == len(tracks)
    with pytest.raises(ValueError, match="one result set per tile"):
        ukf.run_many(tiles, results[:-1])
    del results
    torch.cuda.empty_cache()


def test_pipelined_host_output_sets(cuda, native_lib):
    """run_host_pipelined over three equal-shape pinned tiles, per output set: every host buffer equals the view or gather
    of a plain device run of that tile; mismatched tile shapes and output sets raise."""
    import torch

    from ship_track_estimators_b200.batch_n import BatchedUKFN
    from ship_track_estimators_b200.performance_metrics import track_metrics

    ukf = BatchedUKFN(H5, Q5, R5, P5)
    dev_tiles = [_synthetic_tile(80 + j) for j in range(3)]
    full = [ukf.run(t) for t in dev_tiles]
    pinned = [t.pin_memory() for t in dev_tiles]
    diag = [0, 6, 12, 18, 24]
    for name, keys in ukf.OUTPUT_SETS.items():
        outs = [ukf.host_outputs(pinned[0], outputs=name) for _ in pinned]
        moved = ukf.run_host_pipelined(pinned, outs, device=cuda, outputs=name)
        torch.cuda.synchronize()
        assert moved["d2h_bytes"] == sum(v.numel() * v.element_size() for o in outs for v in o.values())
        assert moved["h2d_bytes"] == sum(p.input_bytes() for p in pinned)
        for j, (o, f, t) in enumerate(zip(outs, full, dev_tiles)):
            assert torch.equal(o["status"], f.status.cpu()) and torch.equal(o["n_updates"], f.n_updates.cpu())
            nsteps = torch.from_numpy(t.n_steps_host.astype(np.int64))
            valid = (torch.arange(f.mean_f.shape[0])[:, None, None] <= nsteps[None, None, :]).double()   # rows a track wrote
            for key in keys:
                if key in ("mean_f", "cov_f", "mean_s", "cov_s"):
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
                assert torch.equal(torch.nan_to_num(o[key]) * w, torch.nan_to_num(want) * w), (name, key, j)
    # the same tiles through run_host, one at a time, into a host TrackResultsN
    host = full[0].host_like()
    moved = ukf.run_host(pinned[0], host, device=cuda)
    torch.cuda.synchronize()
    assert moved["d2h_bytes"] == sum(getattr(host, n).numel() * 8 for n in ("mean_f", "cov_f", "mean_s", "cov_s")) + 8 * len(host.status)
    assert torch.equal(host.status, full[0].status.cpu()) and torch.equal(host.n_updates, full[0].n_updates.cpu())
    nsteps = torch.from_numpy(dev_tiles[0].n_steps_host.astype(np.int64))
    valid = (torch.arange(host.mean_f.shape[0])[:, None, None] <= nsteps[None, None, :]).double()
    for key in ("mean_f", "cov_f", "mean_s", "cov_s"):
        assert torch.equal(torch.nan_to_num(getattr(host, key)) * valid, torch.nan_to_num(getattr(full[0], key).cpu()) * valid), key
    other = _synthetic_tile(90, T=128).pin_memory()
    with pytest.raises(ValueError, match="share one shape"):
        ukf.run_host_pipelined([pinned[0], other], [ukf.host_outputs(pinned[0]), ukf.host_outputs(other)], device=cuda)
    with pytest.raises(ValueError, match="one host output set per tile"):
        ukf.run_host_pipelined(pinned, [ukf.host_outputs(pinned[0])], device=cuda)
    with pytest.raises(ValueError, match="needs the smoother"):
        ukf.run_host_pipelined(pinned, [{} for _ in pinned], device=cuda, outputs="cli", smoother=False)
    with pytest.raises(ValueError, match="unknown output"):
        ukf.run_host_pipelined(pinned, [{} for _ in pinned], device=cuda, outputs=("cov_f", "gate_iters"))


def test_local_summary_of_five_state_results(cuda, native_lib):
    import torch

    from ship_track_estimators_b200.batch_n import BatchedUKFN
    from ship_track_estimators_b200.sharding import local_summary

    b = _synthetic_tile(95)
    res = BatchedUKFN(H5, Q5, R5, P5).run(b)
    s = local_summary(res, b.track_steps())
    assert s["tracks"] == b.n_tracks and s["track_steps"] == float(b.n_steps_host.sum())
    assert s["updates"] == float(res.n_updates.sum()) and s["flagged"] == float((res.status != 0).sum())
    assert s["checksum"] == float(torch.nan_to_num(res.mean_s[0]).sum())


def test_estimate_fleet_dim5_writes_the_class_api_files(cuda, native_lib, tmp_path):
    """estimate_fleet with a five-state input.json: every file of every ship byte-identical to write_track_outputs of
    UnscentedKalmanFilter(..., non_linear_process=geodetic_dynamics_turn) run + run_rts_smoother on that ship's CLI
    measurements (derived on the device, zero-padded to five rows); the same files when the fleet is cut into tiles."""
    from test_host_dropin import _fleet_csv

    from ship_track_estimators_b200.cli.writers import estimate_fleet, write_track_outputs
    from ship_track_estimators_b200.kalman_filters import UnscentedKalmanFilter, geodetic_dynamics_turn
    from ship_track_estimators_b200.utils import generate_dts

    csv = str(tmp_path / "fleet.csv")
    _fleet_csv(csv, seed=33, n_ships=36, time_ordered=True)
    settings = {"dim": 5, "H": [1, 1, 0, 0, 0], "R": [0.001, 0.001, 0, 0, 0], "Q": [1e-2, 1e-2, 1e-4, 1e-4, 1e-5],
                "P": [1.0, 1.0, 1.0, 4.0, 1e-2], "dt": -1, "nsteps": 2, "smooth": 2}
    kw = dict(id_col="primary.id", lat_col="lat", lon_col="lon", apply_rts_smoother=True, device=cuda)
    one, tiled, ref = (str(tmp_path / d) for d in ("one", "tiled", "ref"))
    for d in (one, tiled, ref):
        os.makedirs(d)
    fleet, res = estimate_fleet(csv, settings, directory=one, **kw)
    assert fleet.n_tracks >= 20 and res is not None and res.mean_f.shape[1] == 5
    fleet_t, res_t = estimate_fleet(csv, settings, directory=tiled, tile_plan=dict(state_budget=400, granule=4), **kw)
    assert res_t is None and fleet_t.ids == fleet.ids

    H, Q, R, P = (np.diag(np.asarray(settings[k], dtype=np.float64)) for k in ("H", "Q", "R", "P"))
    b4 = fleet.to_batch(device=cuda, substeps=2, smooth_width=2, need_rows=(True,) * 4, geodesy="wgs84")
    col_of = np.arange(fleet.n_tracks) if b4.order is None else np.argsort(b4.order)
    rows = [r.cpu().numpy() for r in b4.z]
    sr, cr = b4.sog_rate.cpu().numpy(), b4.cog_rate.cpu().numpy()
    for i, sid in enumerate(fleet.ids):
        lat, lon, dts = fleet.track(i)
        j, m = int(col_of[i]), int(fleet.n_obs[i])
        st = SimpleNamespace(dts=dts, z=np.stack([r[:m, j] for r in rows]), sog_rate=sr[:m, j], cog_rate=cr[:m, j])
        dt = generate_dts(dts, 2)
        ukf = UnscentedKalmanFilter(H=H, Q=Q, R=R, P=P, x0=np.append(st.z[:, 0], 0.0), non_linear_process=geodetic_dynamics_turn,
                                    noise="zero")
        means, covs = ukf.run(len(dt), dt, st)
        means_s, covs_s = ukf.run_rts_smoother(st)
        write_track_outputs("output", sid, means, covs, dt, lon, lat, means_s, covs_s, ref)
    names = sorted(os.listdir(ref))
    assert len(names) == 6 * fleet.n_tracks and sorted(os.listdir(one)) == names and sorted(os.listdir(tiled)) == names
    for name in names:
        want = open(os.path.join(ref, name), "rb").read()
        assert open(os.path.join(one, name), "rb").read() == want, name
        assert open(os.path.join(tiled, name), "rb").read() == want, name
    assert np.loadtxt(os.path.join(one, f"output_{fleet.ids[0]}_predictions.txt")).shape[1] == 5
