"""Output side of the CLI: the text files ``track_estimator`` writes (``main_cli.py:146-167``), for one
ship or for a whole fleet processed in one batch (SURVEY.md section 8(f), row N3)."""
from __future__ import annotations

import os
import time
from concurrent.futures import ThreadPoolExecutor
from typing import Mapping, Optional, Sequence

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


FORMATTERS = ("host", "device")


def _check_formatter(formatter: str) -> None:
    if formatter not in FORMATTERS:
        raise ValueError(f"formatter must be one of {FORMATTERS}, not {formatter!r}")


def write_fleet_outputs(prefix: str, fleet, results, substeps: int, directory: str = ".", ships: Optional[Sequence[int]] = None,
                        formatter: str = "host", stats: Optional[dict] = None) -> int:
    """The same files for every ship of a fleet filtered in one batch: ``fleet`` an
    :class:`~ship_track_estimators_b200.ingest.FleetFixes`, ``results`` the
    :class:`~ship_track_estimators_b200.batch.TrackResults` (or five-state ``batch_n.TrackResultsN``) of the tile
    built from it with ``substeps`` predicts per gap.  Returns the number of files written.

    ``formatter="host"`` writes each file with ``np.savetxt``.  ``formatter="device"`` formats the text of every file on
    the GPU (``text.format_tables``), copies it to pinned host memory once per chunk of ships and writes each file with
    one ``write`` from a small thread pool while the next chunk formats; the files are byte-identical.  It needs results
    on a CUDA device.  ``stats``, if given, receives the device path's timings: ``format_s`` (kernels and scan),
    ``copy_s`` (device to host), ``write_s`` (seconds spent in file writes, summed over the writer threads), ``bytes``."""
    _check_formatter(formatter)
    if formatter == "device":
        return _write_fleet_outputs_device(prefix, fleet, results, substeps, directory, ships, stats)
    from ..utils import generate_dts

    n = 0
    results = results.to_host()   # one device->host transfer per array, not eight small ones per ship
    for i in (range(fleet.n_tracks) if ships is None else ships):
        tr = results.track(i)
        lat, lon, dts = fleet.track(i)
        n += len(write_track_outputs(prefix, fleet.ids[i], tr["means"], tr["covs"], generate_dts(dts, substeps), lon, lat,
                                     tr.get("means_s"), tr.get("covs_s"), directory))
    return n


#: Values formatted per device pass: bounds the scratch (36 B per value) and the text buffers (27 B per value).
CHUNK_VALUES = 1 << 25
_WRITER_THREADS = 8


def _write_files(done_event, buf: np.ndarray, offsets: np.ndarray, paths: list) -> float:
    done_event.synchronize()
    t0 = time.perf_counter()
    mv = memoryview(buf)
    for g, path in enumerate(paths):
        with open(path, "wb") as fh:
            fh.write(mv[offsets[g]:offsets[g + 1]])
    return time.perf_counter() - t0


def _write_fleet_outputs_device(prefix, fleet, results, substeps, directory, ships, stats) -> int:
    import torch

    from ..text import Table, diagonal_planes, format_tables

    if not results.mean_f.is_cuda:
        raise ValueError('formatter="device" formats results that are on a CUDA device; use formatter="host" for host results')
    dev = results.mean_f.device
    ships = np.arange(fleet.n_tracks, dtype=np.int64) if ships is None else np.asarray(list(ships), dtype=np.int64)
    cols = np.array([results.column(int(i)) for i in ships], dtype=np.int64)   # IndexError for a ship the tile does not hold
    n_steps = (np.asarray(results.n_steps_host, dtype=np.int64)[cols] if results.n_steps_host is not None
               else np.full(len(cols), results.mean_f.shape[0] - 1, dtype=np.int64))
    n_obs = np.asarray(fleet.n_obs, dtype=np.int64)[ships]
    ns, diag = results.mean_f.shape[1], diagonal_planes(results.cov_f.shape[1])
    smoothed = results.mean_s is not None
    # per ship, in write_track_outputs' order: predictions, variances, dts, original track[, the two smoothed files]
    rows = [n_steps + 1, n_steps + 1, (n_obs - 1) * substeps if substeps > 0 else 0 * n_obs, n_obs]
    ncols = [ns, ns, 1, 2]
    if smoothed:
        rows += [n_steps + 1, n_steps + 1]
        ncols += [ns, ns]
    n_tables = len(ncols)
    counts = np.stack(rows, axis=1) * np.array(ncols)                  # [ships][tables] values
    if len(ships) == 0:
        return 0
    csum = np.cumsum(counts.sum(axis=1))
    cuts = [0]                                                          # chunks of ships of <= CHUNK_VALUES values (or one ship)
    while cuts[-1] < len(ships):
        before = int(csum[cuts[-1] - 1]) if cuts[-1] else 0
        cuts.append(max(int(np.searchsorted(csum, before + CHUNK_VALUES, side="right")), cuts[-1] + 1))

    with torch.cuda.device(dev):   # kernels, copies and timing events on one stream of the results' device
        pool = ThreadPoolExecutor(max_workers=_WRITER_THREADS)
        pending, timings, n_bytes, write_s = [], [], 0, 0.0
        try:
            for a, b in zip(cuts[:-1], cuts[1:]):
                if len(pending) >= 2:                      # at most two chunks of pinned text in flight
                    write_s += sum(f.result() for f in pending.pop(0))
                idx = ships[a:b]
                m = int(n_obs[a:b].max())
                fix = np.zeros((m, 3, b - a))                                # lon, lat, dts / substeps of the chunk's ships
                fix[:, 0] = fleet.lon[:m, idx]
                fix[:, 1] = fleet.lat[:m, idx]
                if substeps > 0:
                    fix[: m - 1, 2] = fleet.dts[: m - 1, idx] / substeps      # generate_dts: dts / substeps, repeated
                fix_d = torch.from_numpy(fix).to(dev)
                local = torch.arange(b - a, dtype=torch.int32, device=dev)
                col_d = torch.from_numpy(cols[a:b].astype(np.int32)).to(dev)
                tables = [Table(results.mean_f, col_d, range(ns)), Table(results.cov_f, col_d, diag),
                          Table(fix_d, local, [2], row_div=max(substeps, 1)), Table(fix_d, local, [0, 1])]
                if smoothed:
                    tables += [Table(results.mean_s, col_d, range(ns)), Table(results.cov_s, col_d, diag)]
                vs = np.zeros((b - a) * n_tables + 1, dtype=np.int64)
                np.cumsum(counts[a:b].reshape(-1), out=vs[1:])
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                ev[0].record()
                text, offsets = format_tables(tables, torch.from_numpy(vs).to(dev), int(vs[-1]))
                ev[1].record()
                offsets = offsets.cpu().numpy()
                host = torch.empty(int(offsets[-1]), dtype=torch.uint8, pin_memory=True)
                host.copy_(text[: host.numel()], non_blocking=True)
                ev[2].record()
                timings.append(ev)
                n_bytes += host.numel()
                paths = []
                for i in idx:
                    stem = os.path.join(directory, f"{prefix}_{fleet.ids[i]}")
                    paths += [f"{stem}_predictions.txt", f"{stem}_variances.txt", f"{stem}_dts.txt",
                              os.path.join(directory, f"original_{fleet.ids[i]}_track.txt")]
                    if smoothed:
                        paths += [f"{stem}_predictions_smoothed.txt", f"{stem}_variances_smoothed.txt"]
                buf = host.numpy()
                step = -(-len(paths) // _WRITER_THREADS)
                pending.append([pool.submit(_write_files, ev[2], buf, offsets[g:], paths[g:g + step])
                                for g in range(0, len(paths), step)])
            write_s += sum(f.result() for fs in pending for f in fs)
        finally:
            pool.shutdown(wait=True)
    if stats is not None:
        stats.update(format_s=sum(e[0].elapsed_time(e[1]) for e in timings) / 1e3,
                     copy_s=sum(e[1].elapsed_time(e[2]) for e in timings) / 1e3, write_s=write_s, bytes=n_bytes,
                     chunks=len(timings))
    return len(ships) * n_tables


def estimate_fleet(track_file: str, settings: dict, id_col: str = "id", lat_col: str = "lat", lon_col: str = "lon",
                   ship_ids: Optional[Sequence] = None, reverse: bool = False, apply_rts_smoother: bool = False,
                   output_prefix: str = "output", directory: str = ".", device="cuda", geodesy: str = "wgs84", min_fixes: int = 3,
                   tile_plan: Optional[dict] = None, formatter: str = "host", ship_settings: Optional[Mapping[str, Mapping]] = None):
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
    ``results`` is then None.  ``ValueError`` when no ship has ``min_fixes`` fixes.  ``formatter``: that of
    :func:`write_fleet_outputs` (``"device"`` formats the files on the GPU).

    ``ship_settings`` (``dim: 5``) maps a ship id to its own noise, ``{"Q": ..., "R": ...}`` (either or both) in the
    ``input.json`` matrix format: those ships get what the class API gives with that ``Q`` / ``R``, the others the
    file's.  It is checked before any device work: an id the file does not hold or another key raises ``ValueError``,
    a matrix of the wrong dimension what ``input.json`` would raise, an asymmetric one ``ValueError``, and ``dim: 4``
    ``NotImplementedError``."""
    from .main_cli import get_input_settings

    _check_formatter(formatter)
    dim, dt, nsteps, H, Q, R, P, smooth_control = get_input_settings(settings)
    if dim not in (4, 5):
        raise NotImplementedError("the CUDA path implements the 4-state geodetic model and the 5-state turn-rate model")
    overrides = _ship_noise(ship_settings, dim)
    from ..ingest import read_csv_fleet

    fleet = read_csv_fleet(track_file, id_col=id_col, lat_col=lat_col, lon_col=lon_col, ship_ids=ship_ids, reverse=reverse,
                           on_bad_rows="skip")
    unknown = sorted(set(overrides) - set(fleet.ids))
    if unknown:
        raise ValueError(f"ship_settings names ships that are not in {track_file!r}: {unknown}")
    fleet = fleet.select([i for i in range(fleet.n_tracks) if fleet.n_obs[i] >= min_fixes])
    substeps = nsteps if dt in [-1, 0, None] else 1                       # main_cli.py:114-117
    width = smooth_control if smooth_control not in [-1, 0, 1, None] else 0   # main_cli.py:99-104
    if dim == 5:
        return fleet, _estimate_fleet_n5(fleet, H, Q, R, P, substeps, width, apply_rts_smoother, output_prefix, directory, device,
                                         geodesy, tile_plan or {}, formatter, overrides)
    from ..batch import BatchedUKF

    ukf = BatchedUKF(H, Q, R, P)
    batch = fleet.to_batch(device=device, substeps=substeps, smooth_width=width, need_rows=ukf.model.rows_needed(), geodesy=geodesy)
    results = ukf.run(batch, smoother=apply_rts_smoother)
    results.check_status()   # IndexError / FloatingPointError where the per-ship reference run would fail
    write_fleet_outputs(output_prefix, fleet, results, substeps, directory, formatter=formatter)
    return fleet, results


def _ship_noise(ship_settings: Optional[Mapping[str, Mapping]], dim: int) -> dict:
    """``{str(ship id): {"Q": 5 x 5, "R": 5 x 5}}`` (either key) from ``estimate_fleet``'s ``ship_settings``."""
    if not ship_settings:
        return {}
    if dim != 5:
        raise NotImplementedError("ship_settings needs dim: 5; the n = 4 path takes a per-track R through "
                                  "TrackBatch.from_tracks(R=...) but has no per-track Q")
    from ..batch_n import noise_planes
    from .main_cli import _get_input_matrix

    out = {}
    for sid, entry in ship_settings.items():
        extra = sorted(set(entry) - {"Q", "R"})
        if extra:
            raise ValueError(f"ship_settings[{sid!r}]: unknown keys {extra} (per-ship settings take Q and R)")
        mats = {name: _get_input_matrix(entry, name, dim).astype(np.float64) for name in ("Q", "R") if name in entry}
        for name, M in mats.items():
            noise_planes(f"ship_settings[{sid!r}].{name}", [M], 1)   # ValueError unless symmetric
        out[str(sid)] = mats
    return out


def _estimate_fleet_n5(fleet, H, Q, R, P, substeps, width, smoother, prefix, directory, device, geodesy, tile_plan, formatter,
                       overrides):
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
    # per-ship matrices in the fleet's ship order, for the kinds some ship overrides (the others stay shared)
    own = {name: [overrides.get(sid, {}).get(name, M) for sid in fleet.ids] for name, M in (("Q", Q), ("R", R))
           if any(name in o for o in overrides.values())}
    results = None
    for lo, hi in tiles:
        ships = order[lo:hi] if len(tiles) > 1 else None
        part = fleet if ships is None else fleet.select(ships)
        noise = {name: (mats if ships is None else [mats[i] for i in ships]) for name, mats in own.items()}
        res = ukf.run(TrackBatchN.from_batch(part.to_batch(**kw), **noise), smoother=smoother)
        res.check_status()   # IndexError / FloatingPointError where the per-ship reference run would fail
        write_fleet_outputs(prefix, part, res, substeps, directory, formatter=formatter)
        results = res if ships is None else None
    return results
