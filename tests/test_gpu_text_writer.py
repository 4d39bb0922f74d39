"""GPU: the device formatter of the CLI's text files (csrc/ste_text.cu).  The conversion equals CPython's '%.18e' string
for string; write_fleet_outputs(formatter="device") and estimate_fleet(..., formatter="device") write the host writer's
files byte for byte."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _special_values():
    u = lambda bits: np.array(bits, dtype=np.uint64).view(np.float64)   # noqa: E731
    v = [0.0, -0.0, np.inf, -np.inf, np.nan, -np.nan, 5e-324, -5e-324, np.nextafter(2.2250738585072014e-308, 0),
         2.2250738585072014e-308, np.finfo(np.float64).max, -np.finfo(np.float64).max]
    return np.concatenate([np.array(v), u([0x7ff0000000000001, 0xfff0000000000001, 0x7ff8dead0000beef, 0xffffffffffffffff])])


def _conversion_cases():
    rng = np.random.default_rng(20261020)
    parts = [rng.integers(0, 2**64, size=1_000_000, dtype=np.uint64).view(np.float64), _special_values()]
    p10 = []
    for k in range(-323, 309):
        x = float(f"1e{k}")
        p10 += [np.nextafter(x, 0.0), x, np.nextafter(x, np.inf)]
    parts.append(np.array(p10))
    # exact ties: odd m with 3.2e15 <= m < 9e15 times 2^-5 (and other exponents) has 20 significant digits ending in 5
    m = rng.integers(1_600_000_000_000_000, 4_500_000_000_000_000, size=12_000) * 2 + 1
    parts += [m * 2.0 ** -5] + [m[:1000] * 2.0 ** sh for sh in (-1, -2, -3, -4, -6, -7)]
    parts[-7:] = [np.concatenate([p, -p]) for p in parts[-7:]]
    # just below a power of ten: the 19-digit rounding carries into the exponent
    below = []
    for k in range(-300, 301, 3):
        y = float(f"1e{k}")
        for _ in range(8):
            y = np.nextafter(y, 0.0)
            below.append(y)
    parts.append(np.array(below))
    parts += [rng.uniform(-180, 180, 50_000), rng.uniform(-90, 90, 50_000), 10.0 ** rng.uniform(-12, 3, 50_000)]
    return np.concatenate(parts).astype(np.float64)


def test_conversion_matches_cpython_string_for_string(cuda, native_lib):
    import torch

    from ship_track_estimators_b200.text import format_values

    x = _conversion_cases()
    assert len(x) > 1_000_000
    got = format_values(torch.from_numpy(x).to(cuda)).decode("ascii")
    want = "".join("%.18e\n" % v for v in x)
    if got != want:
        g, w = got.split("\n"), want.split("\n")
        bad = [i for i in range(min(len(g), len(w))) if g[i] != w[i]][:5]
        pytest.fail(f"{len(bad)}+ mismatches, first: " + "; ".join(f"{x[i]!r}: {g[i]} != {w[i]}" for i in bad))


def _fleet(seed, T=37):
    from ship_track_estimators_b200.ingest import FleetFixes

    rng = np.random.default_rng(seed)
    n_obs = rng.integers(3, 31, size=T).astype(np.int32)
    n_obs[5] = 2                                          # a ship with two fixes
    m = int(n_obs.max())
    lon = np.cumsum(rng.normal(0, 0.02, (m, T)), axis=0) + rng.uniform(-170, 170, T)
    lat = np.cumsum(rng.normal(0, 0.02, (m, T)), axis=0) + rng.uniform(-60, 60, T)
    dts = rng.choice([0.5, 1.0, 1.5, 3.0], size=(m - 1, T))
    for t in range(T):
        lon[n_obs[t]:, t] = lat[n_obs[t]:, t] = 0.0
        dts[n_obs[t] - 1:, t] = 0.0
    return FleetFixes([f"{100000 + 7 * t}" for t in range(T)], lon, lat, dts, n_obs)


def _same_files(a, b):
    names = sorted(os.listdir(a))
    assert names and names == sorted(os.listdir(b))
    for n in names:
        assert open(os.path.join(a, n), "rb").read() == open(os.path.join(b, n), "rb").read(), n


def _write_both(tmp_path, tag, fleet, res, substeps, ships=None):
    from ship_track_estimators_b200.cli.writers import write_fleet_outputs

    dirs = [str(tmp_path / f"{tag}_{f}") for f in ("host", "device")]
    counts = []
    for d, f in zip(dirs, ("host", "device")):
        os.makedirs(d)
        counts.append(write_fleet_outputs("out", fleet, res, substeps, d, ships=ships, formatter=f))
    assert counts[0] == counts[1] == len(os.listdir(dirs[0]))
    _same_files(*dirs)
    return dirs


@pytest.mark.parametrize("packed", [False, True])
@pytest.mark.parametrize("smoother", [False, True])
@pytest.mark.parametrize("substeps", [1, 3])
def test_fleet_files_n4_byte_identical(packed, smoother, substeps, cuda, native_lib, tmp_path):
    from ship_track_estimators_b200.batch import BatchedUKF

    fleet = _fleet(10 + substeps)
    H, R = np.diag([1.0, 1.0, 0.0, 0.0]), np.diag([1e-3, 1e-3, 0.0, 0.0])
    ukf = BatchedUKF(H, np.diag([1e-2, 1e-2, 1e-4, 1e-4]), R, np.eye(4), packed_cov=packed)
    res = ukf.run(fleet.to_batch(device=cuda, substeps=substeps, need_rows=ukf.model.rows_needed()), smoother=smoother)
    assert res.order is not None and res.packed_cov == packed
    host, _ = _write_both(tmp_path, "all", fleet, res, substeps)
    assert len(os.listdir(host)) == fleet.n_tracks * (6 if smoother else 4)
    _write_both(tmp_path, "some", fleet, res, substeps, ships=[5, 30, 2, 11])


def test_fleet_files_n5_byte_identical(cuda, native_lib, tmp_path):
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    fleet = _fleet(21)
    d5 = np.diag
    ukf = BatchedUKFN(d5([1.0, 1, 0, 0, 0]), d5([1e-2, 1e-2, 1e-4, 1e-4, 1e-5]), d5([1e-3, 1e-3, 0, 0, 0]), d5([1.0, 1, 1, 4, 1e-2]))
    res = ukf.run(TrackBatchN.from_batch(fleet.to_batch(device=cuda, substeps=2, need_rows=(True,) * 4)), smoother=True)
    _write_both(tmp_path, "n5", fleet, res, 2)
    _write_both(tmp_path, "n5some", fleet, res, 2, ships=[36, 0, 5])


def test_order_independence(cuda, native_lib, tmp_path):
    """The same fleet twice, and packed in another column order, gives the same files."""
    from ship_track_estimators_b200.batch import BatchedUKF
    from ship_track_estimators_b200.cli.writers import write_fleet_outputs

    fleet = _fleet(5)
    ukf = BatchedUKF(np.diag([1.0, 1, 0, 0]), np.diag([1e-2, 1e-2, 1e-4, 1e-4]), np.diag([1e-3, 1e-3, 0, 0]), np.eye(4))
    runs = [(ukf.run(fleet.to_batch(device=cuda, substeps=2, need_rows=ukf.model.rows_needed(), sort_by_length=s), smoother=True))
            for s in (True, True, False)]
    assert runs[0].order is not None and runs[2].order is None
    dirs = []
    for j, res in enumerate(runs):
        dirs.append(str(tmp_path / f"run{j}"))
        os.makedirs(dirs[-1])
        write_fleet_outputs("out", fleet, res, 2, dirs[-1], formatter="device")
    _same_files(dirs[0], dirs[1])
    _same_files(dirs[0], dirs[2])


@pytest.mark.parametrize("dim", [4, 5])
def test_estimate_fleet_device_formatter(dim, cuda, native_lib, tmp_path):
    from test_host_dropin import _fleet_csv

    from ship_track_estimators_b200.cli.writers import estimate_fleet

    csv = str(tmp_path / "fleet.csv")
    _fleet_csv(csv, seed=34, n_ships=30, time_ordered=True)
    z = [0] * (dim - 4)
    settings = {"dim": dim, "H": [1, 1, 0, 0] + z, "R": [0.001, 0.001, 0, 0] + z, "Q": [1e-2, 1e-2, 1e-4, 1e-4] + [1e-5] * (dim - 4),
                "P": [1.0, 1.0, 1.0, 4.0] + [1e-2] * (dim - 4), "dt": -1, "nsteps": 2, "smooth": 2}
    kw = dict(id_col="primary.id", lat_col="lat", lon_col="lon", apply_rts_smoother=True, device=cuda)
    if dim == 5:
        kw["tile_plan"] = dict(state_budget=400, granule=4)   # several tiles
    dirs = {}
    for f in ("host", "device"):
        dirs[f] = str(tmp_path / f)
        os.makedirs(dirs[f])
        fleet, res = estimate_fleet(csv, settings, directory=dirs[f], formatter=f, **kw)
    assert fleet.n_tracks >= 20 and (res is None) == (dim == 5)
    assert len(os.listdir(dirs["host"])) == 6 * fleet.n_tracks
    _same_files(dirs["host"], dirs["device"])


def test_results_on_another_device_than_the_current_one(native_lib, tmp_path):
    """Results on the last visible GPU while cuda:0 is current: the kernels, the scan and the copy run on the results'
    device and the files equal the host writer's."""
    import torch

    from ship_track_estimators_b200.batch import BatchedUKF

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    dev = torch.device(f"cuda:{torch.cuda.device_count() - 1}")
    fleet = _fleet(6)
    ukf = BatchedUKF(np.diag([1.0, 1, 0, 0]), np.diag([1e-2, 1e-2, 1e-4, 1e-4]), np.diag([1e-3, 1e-3, 0, 0]), np.eye(4))
    res = ukf.run(fleet.to_batch(device=dev, substeps=2, need_rows=ukf.model.rows_needed()), smoother=True)
    assert res.mean_f.device == dev
    with torch.cuda.device(0):
        _write_both(tmp_path, "other", fleet, res, 2)
