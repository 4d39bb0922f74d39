"""CPU: the host-side drop-ins around the hot path (ShipTrack ingest, CLI parsing, JSON settings).
Known answers: SURVEY.md section 9.3 (generated from the reference) and the golden fixture of
BASELINE config 1, whose derived inputs were produced by the reference's own ShipTrack."""
import json
import os

import numpy as np
import pandas as pd
import pytest

from _helpers import REPO, load_golden
from ship_track_estimators_b200.cli.argument_parser import create_parser
from ship_track_estimators_b200.cli.main_cli import _get_input_matrix, get_input_settings
from ship_track_estimators_b200.ship_track import ShipTrack
from ship_track_estimators_b200.utils import haversine_formula, heading


def write_track_csv(path, ship_id, lon, lat, dts_hours, id_col="primary.id", extra_rows=()):
    """A CSV in the reference's data format (yr, mo, dy, hr columns) for the given fixes."""
    when = pd.Timestamp("1880-03-01") + pd.to_timedelta(np.concatenate(([0.0], np.cumsum(dts_hours))), unit="h")
    rows = [dict(**{id_col: ship_id}, yr=d.year, mo=d.month, dy=d.day, hr=d.hour, lat=la, lon=lo) for d, lo, la in zip(when, lon, lat)]
    rows[1:1] = list(extra_rows)
    # like the reference's historical file, the id column also holds a non-numeric value (there: an
    # embedded header row), which keeps pandas from parsing ids such as "01203823" as integers
    rows.append(dict(**{id_col: "id.tidy"}, yr=1880, mo=1, dy=1, hr=0, lat=0.0, lon=0.0))
    pd.DataFrame(rows).to_csv(path, index=False)


def test_ship_track_known_answers(tmp_path):
    lon = [-30.5, -31.5, -32.5, -33.5, -33.5]; lat = [-0.5, -3.5, -6.5, -8.5, -11.5]
    csv = str(tmp_path / "t.csv")
    write_track_csv(csv, "A7", lon, lat, [24, 24, 24, 12], id_col="id",
                    extra_rows=[dict(id="other", yr=1880, mo=1, dy=1, hr=3, lat=1.0, lon=2.0)])
    st = ShipTrack(calc_distance_func=haversine_formula, calc_heading_func=heading)
    out = st.read_csv(csv, ship_id="A7")
    assert out[0] is st.lat and np.array_equal(st.dts, [24.0, 24.0, 24.0, 12.0]) and len(st.dates) == 5
    z = st.get_measurements(include_sog=True, include_cog=True)
    st.calculate_cog_rate(); st.calculate_sog_rate()
    assert z.shape == (4, 5) and np.array_equal(z[0], lon)
    np.testing.assert_allclose(st.sog, [14.666569517825678, 14.66188856000385, 10.35378642995031, 27.829872698318386, 27.829872698318386], rtol=1e-14)
    np.testing.assert_allclose(st.cog, [198.40941994487474, 198.32831442189988, 206.30510826660182, 180, 180], rtol=1e-14)
    np.testing.assert_allclose(st.sog_rate, [0, -1.9503990924281864e-04, -1.7950425541889756e-01, 7.2817026118200323e-01, 0], rtol=1e-10)
    np.testing.assert_allclose(st.cog_rate, [0, -0.00337939679061942, 0.33236641019591434, -1.0960461777750758, 0], rtol=1e-10)
    assert st.get_measurements().shape == (2, 5)
    rev = ShipTrack(calc_distance_func=haversine_formula, calc_heading_func=heading)
    rev.read_csv(csv, ship_id="A7", reverse=True)
    assert np.array_equal(rev.lon, lon[::-1]) and np.array_equal(rev.dts, [12.0, 24.0, 24.0, 24.0])
    with pytest.raises(ValueError, match="No data found"):
        ShipTrack().read_csv(csv, ship_id="nobody")


def test_ship_track_reproduces_reference_derived_inputs(tmp_path):
    """BASELINE config 1 (ship 01203823): rebuilding the CSV rows from the fixture and ingesting
    them gives the z / rates the reference's ShipTrack produced."""
    tr = load_golden("c1_single_ship")[0][0]
    csv = str(tmp_path / "ship.csv")
    write_track_csv(csv, "01203823", tr["z"][0], tr["z"][1], tr["dts"])
    st = ShipTrack(calc_distance_func=haversine_formula, calc_heading_func=heading)
    st.read_csv(csv, ship_id="01203823", id_col="primary.id")
    z = st.get_measurements(include_sog=True, include_cog=True)
    st.calculate_cog_rate(); st.calculate_sog_rate()
    np.testing.assert_allclose(st.dts, tr["dts"], rtol=0, atol=0)
    np.testing.assert_allclose(z, tr["z"], rtol=1e-13)
    np.testing.assert_allclose(st.sog_rate, tr["sog_rate"], rtol=1e-9, atol=1e-13)
    np.testing.assert_allclose(st.cog_rate, tr["cog_rate"], rtol=1e-9, atol=1e-13)


def test_cli_flags_and_settings(tmp_path):
    args = create_parser().parse_args(["-t", "d.csv", "-s", "01203823", "-ic", "primary.id", "-lat", "lat", "-lon", "lon", "-rts"])
    assert (args.input_file, args.output_prefix, args.track_file, args.ship_id) == ("input.json", "output", "d.csv", "01203823")
    assert args.apply_rts_smoother and not args.reverse and args.id_col == "primary.id" and args.lat_id == "lat"
    with pytest.raises(SystemExit):
        create_parser().parse_args(["-s", "x"])  # -t is required
    cfg = {"dim": 4, "H": [1, 1, 0, 0], "R": [0.001, 0.001, 0, 0], "Q": [1e-2, 1e-2, 1e-4, 1e-4], "P": [1.0, 1.0, 1.0, 1.0], "dt": -1, "nsteps": 2}
    dim, dt, nsteps, H, Q, R, P, sm = get_input_settings(cfg)
    assert (dim, dt, nsteps, sm) == (4, -1, 2, None)
    assert np.array_equal(H, np.diag([1, 1, 0, 0])) and np.array_equal(R, np.diag([0.001, 0.001, 0, 0]))
    full = dict(cfg, P=np.eye(4).tolist(), smooth=2)
    assert np.array_equal(get_input_settings(full)[6], np.eye(4)) and get_input_settings(full)[7] == 2
    for missing in ("dim", "dt", "nsteps", "H"):
        with pytest.raises(KeyError):
            get_input_settings({k: v for k, v in cfg.items() if k != missing})
    with pytest.raises(AssertionError):
        _get_input_matrix({"H": [1, 1, 0]}, "H", 4)
    with pytest.raises(AssertionError):
        _get_input_matrix({"H": [[1, 0], [0, 1], [0, 0], [0, 0]]}, "H", 4)
    p = tmp_path / "input.json"
    p.write_text(json.dumps(cfg))
    from ship_track_estimators_b200.cli.json_loader import load_input_json

    assert load_input_json(str(p)) == cfg


def _fleet_csv(path, seed=3, n_ships=9, string_labels=True, time_ordered=False):
    """A file shaped like the historical data: ships interleaved, a leading label column that pandas
    turns into the index, and (optionally) a stray repeated-header row that makes the labels strings."""
    rng = np.random.default_rng(seed)
    rows = []
    for s in range(n_ships):
        n = 1 if s == 0 else int(rng.integers(2, 40))     # one ship with a single fix
        t = pd.Timestamp("1901-03-01") + pd.to_timedelta(np.cumsum(rng.choice([6, 12, 24, 30], n)), unit="h")
        lat = rng.uniform(-50, 50) + np.cumsum(rng.normal(0, 0.3, n))      # a slow random walk: a plausible ship
        lon = rng.uniform(-170, 170) + np.cumsum(rng.normal(0, 0.3, n))
        for j in range(n):
            rows.append({"primary.id": f"0{120000 + s * 7}", "yr": t[j].year, "mo": t[j].month, "dy": t[j].day, "hr": t[j].hour,
                         "lat": round(float(lat[j]), 2), "lon": round(float(lon[j]), 2)})
    order = rng.permutation(len(rows))
    labels = rng.permutation(np.arange(90, 90 + len(rows)))        # labels cross a digit boundary: '100' < '99' as strings
    if time_ordered:    # ships still interleaved, but label order inside a ship follows time (usable tracks)
        order = np.asarray(sorted(range(len(rows)), key=lambda k: (pd.Timestamp(year=rows[k]["yr"], month=rows[k]["mo"],
                                                                                  day=rows[k]["dy"], hour=rows[k]["hr"]), k)))
        labels = np.asarray([f"{k:05d}" for k in range(len(rows))])
    lines = ["primary.id,yr,mo,dy,hr,lat,lon"]                      # header has one column fewer than the rows -> index
    for lab, k in zip(labels, order):
        r = rows[k]
        lines.append(f"{lab},{r['primary.id']},{r['yr']},{r['mo']},{r['dy']},{r['hr']},{r['lat']},{r['lon']}")
        if string_labels and lab == labels[5]:
            lines.append("row,id.tidy,yr,mo,dy,hr,lat,lon")
    with open(path, "w") as fh:
        fh.write("\n".join(lines) + "\n")
    return sorted({r["primary.id"] for r in rows})


@pytest.mark.parametrize("string_labels", [True, False])
def test_bulk_csv_ingest_matches_per_ship_reader(tmp_path, string_labels):
    """ingest.read_csv_fleet (one parse, SoA layout) == ShipTrack.read_csv ship by ship: row selection,
    sort_index order inside a ship (lexicographic when the labels are strings), gaps in hours,
    reverse, explicit id lists, stray rows."""
    from ship_track_estimators_b200.ingest import read_csv_fleet

    csv = str(tmp_path / "fleet.csv")
    ids = _fleet_csv(csv, string_labels=string_labels)
    if not string_labels:
        ids = sorted(str(int(i)) for i in ids)      # an all-numeric id column is parsed as integers (both readers)
    kw = dict(id_col="primary.id", lat_col="lat", lon_col="lon")
    if string_labels:
        with pytest.raises(ValueError, match="unparsable"):
            read_csv_fleet(csv, **kw)
    fleet = read_csv_fleet(csv, on_bad_rows="skip", **kw)
    assert sorted(fleet.ids) == ids and fleet.lon.shape == (int(fleet.n_obs.max()), len(ids))
    for reverse in (False, True):
        fl = read_csv_fleet(csv, ship_ids=ids[::-1], reverse=reverse, **kw)
        assert fl.ids == ids[::-1]
        for i, sid in enumerate(fl.ids):
            lat, lon, dts = ShipTrack().read_csv(csv, ship_id=sid, reverse=reverse, **kw)
            a, b, c = fl.track(i)
            assert np.array_equal(a, lat) and np.array_equal(b, lon) and np.array_equal(c, dts), (sid, reverse)
            assert not fl.lon[len(lat):, i].any() and not fl.dts[max(len(lat) - 1, 0):, i].any()   # zero padding
    with pytest.raises(ValueError, match="No data found"):
        read_csv_fleet(csv, ship_ids=["nobody"], **kw)
    two_plus = [i for i in range(fleet.n_tracks) if fleet.n_obs[i] >= 2]
    assert len(two_plus) == fleet.n_tracks - 1 and fleet.select(two_plus).n_tracks == len(two_plus)
    with pytest.raises(ValueError, match="at least two fixes"):
        fleet.to_batch(device="cpu")


def _historical_csv(path, tracks, ids, seed=5):
    """The layout of the reference's data/historical_ships file (a leading row-label column that pandas turns into the
    index, ships interleaved, an embedded repeated header row whose id is "id.tidy", ``lon2`` beside ``lon``) holding
    the fixes of the committed real ships."""
    rng = np.random.default_rng(seed)
    rows = []
    for s, (tr, sid) in enumerate(zip(tracks, ids)):
        when = pd.Timestamp("1880-01-01") + pd.Timedelta(hours=24 * s) + pd.to_timedelta(np.concatenate(([0.0], np.cumsum(tr["dts"]))), unit="h")
        rows += [(sid, d, float(lo), float(la)) for d, lo, la in zip(when, tr["z"][0], tr["z"][1])]
    order = rng.permutation(len(rows))
    # labels follow file order; zero-padded, so their string order (the header row makes them strings) is their number order
    order = order[np.argsort([rows[k][1] for k in order], kind="stable")]
    lines = ["primary.id,yr,mo,dy,hr,lat,lon,lon2"]
    for lab, k in enumerate(order):
        sid, d, lo, la = rows[k]
        lines.append(f"{lab:05d},{sid},{d.year},{d.month},{d.day},{d.hour},{la!r},{lo!r},{lo!r}")
        if lab == 1:
            lines.append("row,id.tidy,yr,mo,dy,hr,lat,lon,lon2")
    with open(path, "w") as fh:
        fh.write("\n".join(lines) + "\n")


def test_bulk_csv_ingest_on_the_historical_file(tmp_path):
    """The 71 runnable ships of the reference's historical file (fixture c2_historical_batch: fixes and gaps as the
    reference's ShipTrack read them) written back in that file's layout: the bulk reader, the per-ship reader and the
    reference's own readings agree ship by ship."""
    from ship_track_estimators_b200.ingest import read_csv_fleet

    tracks, extra = load_golden("c2_historical_batch")
    ids = [str(i) for i in extra["ids"]]
    csv = str(tmp_path / "historical_ship_data.csv")
    _historical_csv(csv, tracks, ids)
    kw = dict(id_col="primary.id", lat_col="lat", lon_col="lon2")
    fleet = read_csv_fleet(csv, on_bad_rows="skip", **kw)
    assert fleet.n_tracks == len(ids) == 71 and sorted(fleet.ids) == sorted(ids)
    for i in range(fleet.n_tracks):
        lat, lon, dts = ShipTrack().read_csv(csv, ship_id=fleet.ids[i], **kw)
        a, b, c = fleet.track(i)
        assert np.array_equal(a, lat) and np.array_equal(b, lon) and np.array_equal(c, dts)
        tr = tracks[ids.index(fleet.ids[i])]
        assert np.array_equal(b, tr["z"][0]) and np.array_equal(a, tr["z"][1]) and np.array_equal(c, tr["dts"])


def test_reference_import_name_is_an_alias():
    """`track_estimators` (the reference's import name, pyproject.toml packages) serves the same module
    objects as ship_track_estimators_b200; the console script entry point exists."""
    import importlib
    import subprocess
    import sys

    code = (
        "import track_estimators, ship_track_estimators_b200 as impl\n"
        "from track_estimators.kalman_filters.unscented import UnscentedKalmanFilter\n"
        "from track_estimators.kalman_filters.non_linear_process import geodetic_dynamics\n"
        "from track_estimators.kalman_filters.kalman_filter import KalmanFilterBase\n"
        "from track_estimators.ship_track import ShipTrack\n"
        "from track_estimators.utils import generate_dts, smooth, haversine_formula, heading\n"
        "from track_estimators.cli.main_cli import track_estimator\n"
        "import ship_track_estimators_b200.kalman_filters.unscented as u\n"
        "assert UnscentedKalmanFilter is u.UnscentedKalmanFilter and issubclass(UnscentedKalmanFilter, KalmanFilterBase)\n"
        "assert track_estimators.utils is impl.utils if hasattr(impl, 'utils') else True\n"
        "try:\n"
        "    import track_estimators.gaussian_processes\n"
        "except ImportError:\n"
        "    print('ok')\n"
    )
    # a fresh interpreter: other tests may have put the real reference on sys.path under the same name
    out = subprocess.run([sys.executable, "-c", code], cwd=REPO, capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stderr
    import tomllib

    with open(os.path.join(REPO, "pyproject.toml"), "rb") as fh:
        meta = tomllib.load(fh)
    assert meta["project"]["scripts"]["track_estimator"] == "ship_track_estimators_b200.cli.main_cli:track_estimator"
    mod, fn = meta["project"]["scripts"]["track_estimator"].split(":")
    assert callable(getattr(importlib.import_module(mod), fn))
