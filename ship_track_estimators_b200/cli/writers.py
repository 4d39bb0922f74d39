"""Output side of the CLI: the text files ``track_estimator`` writes (``main_cli.py:146-167``), for one
ship or for a whole fleet processed in one batch (SURVEY.md section 8(f), row N3)."""
from __future__ import annotations

import os
from typing import Optional, Sequence

import numpy as np


def write_track_outputs(prefix: str, ship_id, means, covs, dt_array, lon, lat, means_s=None, covs_s=None,
                        directory: str = ".") -> list:
    """The reference's files for one ship: ``{prefix}_{id}_predictions.txt`` (states, one row per
    filter state), ``_variances.txt`` (diagonals of the covariances), ``_dts.txt``,
    ``original_{id}_track.txt`` (lon, lat of the fixes) and, with smoothed results, the two
    ``*_smoothed.txt`` files - all through ``np.savetxt`` with its default format."""
    stem = os.path.join(directory, f"{prefix}_{ship_id}")
    out = [(f"{stem}_predictions.txt", np.asarray(means)),
           (f"{stem}_variances.txt", np.diagonal(np.asarray(covs), axis1=1, axis2=2)),
           (f"{stem}_dts.txt", np.asarray(dt_array)),
           (os.path.join(directory, f"original_{ship_id}_track.txt"), np.array((lon, lat)).T)]
    if means_s is not None:
        out += [(f"{stem}_predictions_smoothed.txt", np.asarray(means_s)),
                (f"{stem}_variances_smoothed.txt", np.diagonal(np.asarray(covs_s), axis1=1, axis2=2))]
    for path, arr in out:
        np.savetxt(path, arr)
    return [p for p, _ in out]


def write_fleet_outputs(prefix: str, fleet, results, substeps: int, directory: str = ".", ships: Optional[Sequence[int]] = None) -> int:
    """The same files for every ship of a fleet filtered in one batch: ``fleet`` an
    :class:`~ship_track_estimators_b200.ingest.FleetFixes`, ``results`` the
    :class:`~ship_track_estimators_b200.batch.TrackResults` (or five-state ``batch_n.TrackResultsN``) of the tile
    built from it with ``substeps`` predicts per gap.  Returns the number of files written."""
    from ..utils import generate_dts

    n = 0
    results = results.to_host()   # one device->host transfer per array, not eight small ones per ship
    for i in (range(fleet.n_tracks) if ships is None else ships):
        tr = results.track(i)
        lat, lon, dts = fleet.track(i)
        n += len(write_track_outputs(prefix, fleet.ids[i], tr["means"], tr["covs"], generate_dts(dts, substeps), lon, lat,
                                     tr.get("means_s"), tr.get("covs_s"), directory))
    return n


def estimate_fleet(track_file: str, settings: dict, id_col: str = "id", lat_col: str = "lat", lon_col: str = "lon",
                   ship_ids: Optional[Sequence] = None, reverse: bool = False, apply_rts_smoother: bool = False,
                   output_prefix: str = "output", directory: str = ".", device="cuda", geodesy: str = "wgs84", min_fixes: int = 3,
                   tile_plan: Optional[dict] = None):
    """``track_estimator`` for every ship of a CSV at once: one parse (``ingest.read_csv_fleet``), SOG /
    COG / rates on the device (the CLI's default WGS84 pair, its box smoothing), one filter launch and
    one smoother launch for the whole fleet, then the CLI's files per ship.  ``settings`` is the
    ``input.json`` dictionary.  Ships with fewer than ``min_fixes`` fixes are left out.  Returns
    ``(fleet, results)``.

    ``dim: 5`` runs the five-state turn-rate model (``geodetic_dynamics_turn``, 5 x 5 ``H``, ``Q``, ``R``,
    ``P``): every ship gets what ``UnscentedKalmanFilter(H, Q, R, P, x0, non_linear_process=geodetic_dynamics_turn)``
    gives with ``run`` (+ ``run_rts_smoother``) on the CLI's measurements zero-padded to five rows (the turn rate
    starts at 0 and is not observed), and the files have five columns.  A fleet larger than one five-state tile
    (``batch_n.STATE_BUDGET`` stored states; ``tile_plan``: other keyword arguments of
    ``sharding.plan_ragged_tiles``) runs tile by tile, each tile's files written before the next tile runs;
    ``results`` is then None.  ``ValueError`` when no ship has ``min_fixes`` fixes."""
    from .main_cli import get_input_settings

    dim, dt, nsteps, H, Q, R, P, smooth_control = get_input_settings(settings)
    if dim not in (4, 5):
        raise NotImplementedError("the CUDA path implements the 4-state geodetic model and the 5-state turn-rate model")
    from ..ingest import read_csv_fleet

    fleet = read_csv_fleet(track_file, id_col=id_col, lat_col=lat_col, lon_col=lon_col, ship_ids=ship_ids, reverse=reverse,
                           on_bad_rows="skip")
    fleet = fleet.select([i for i in range(fleet.n_tracks) if fleet.n_obs[i] >= min_fixes])
    substeps = nsteps if dt in [-1, 0, None] else 1                       # main_cli.py:114-117
    width = smooth_control if smooth_control not in [-1, 0, 1, None] else 0   # main_cli.py:99-104
    if dim == 5:
        return fleet, _estimate_fleet_n5(fleet, H, Q, R, P, substeps, width, apply_rts_smoother, output_prefix, directory, device,
                                         geodesy, tile_plan or {})
    from ..batch import BatchedUKF

    ukf = BatchedUKF(H, Q, R, P)
    batch = fleet.to_batch(device=device, substeps=substeps, smooth_width=width, need_rows=ukf.model.rows_needed(), geodesy=geodesy)
    results = ukf.run(batch, smoother=apply_rts_smoother)
    results.check_status()   # IndexError / FloatingPointError where the per-ship reference run would fail
    write_fleet_outputs(output_prefix, fleet, results, substeps, directory)
    return fleet, results


def _estimate_fleet_n5(fleet, H, Q, R, P, substeps, width, smoother, prefix, directory, device, geodesy, tile_plan):
    import numpy as np

    from ..batch_n import STATE_BUDGET, BatchedUKFN, TrackBatchN
    from ..sharding import plan_ragged_tiles

    if fleet.n_tracks == 0:
        raise ValueError("no ship of the file has enough fixes to filter (min_fixes)")
    ukf = BatchedUKFN(H, Q, R, P)
    # Every observation row, whatever H and R reference: the dense five-state update forms z - H x over all rows, and
    # the class API run it must equal gets the CLI's four measured rows.
    kw = dict(device=device, substeps=substeps, smooth_width=width, need_rows=(True,) * 4, geodesy=geodesy)
    order = np.argsort(-fleet.n_obs.astype(np.int64), kind="stable")
    steps = (fleet.n_obs[order].astype(np.int64) - 1) * substeps
    plan = dict(tile_plan)
    tiles = plan_ragged_tiles(steps, plan.pop("state_budget", STATE_BUDGET), **plan)
    results = None
    for lo, hi in tiles:
        ships = order[lo:hi] if len(tiles) > 1 else None
        part = fleet if ships is None else fleet.select(ships)
        res = ukf.run(TrackBatchN.from_batch(part.to_batch(**kw)), smoother=smoother)
        res.check_status()   # IndexError / FloatingPointError where the per-ship reference run would fail
        write_fleet_outputs(prefix, part, res, substeps, directory)
        results = res if ships is None else None
    return results
