"""Choosing a filter's process and measurement noise by maximum likelihood: a grid search over ``(Q, R)`` candidates.

Every candidate is scored on the device by ``BatchedUKF.score`` / ``BatchedUKFN.score``: one store-free forward pass per
(candidate, track) pair that sums the Gaussian log-likelihood of each fix under its one-step prediction
(``performance_metrics.innovation_metrics`` of a run with that candidate, without the run's states).  The largest
summed log-likelihood is the maximum-likelihood choice, for the whole fleet or for each track on its own; the per-track
choice is what ``TrackBatchN.from_tracks(Q=..., R=...)`` takes at n = 5, and ``TrackBatch.from_tracks(Q=..., R=...)`` or
``TrackBatch.with_noise(Q=..., R=...)`` at n = 4.  At n = 4 a per-track ``R`` selects the generic update (as
``TrackBatch.R`` always does), so a grid over ``Q`` alone keeps a position-only filter on its fast update.

    grid = noise_grid(Q, R, q_scales=(0.5, 1, 2), r_scales=(0.25, 0.5, 1, 2, 4))
    fit = fit_noise(engine, TrackBatchN.fleet_tiles(tracks, dts), grid, per="track")
    tiles = TrackBatchN.fleet_tiles(tracks, dts, Q=fit["Q"], R=fit["R"])

    fit = fit_noise(ukf, tile, noise_grid(Q, R, q_scales=(0.25, 0.5, 1, 2, 4), r_scales=(1,)), per="track")   # n = 4
    res = ukf.run(tile.with_noise(Q=fit["Q"]))
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import numpy as np

__all__ = ["noise_grid", "fit_noise", "select_noise"]


def noise_grid(Q, R, q_scales: Sequence[float], r_scales: Sequence[float]) -> List[tuple]:
    """The candidates ``(q * Q, r * R)`` for every ``q`` of ``q_scales`` and ``r`` of ``r_scales``, q-major: candidate
    ``i * len(r_scales) + j`` is ``(q_scales[i] * Q, r_scales[j] * R)``."""
    Q, R = np.asarray(Q, dtype=np.float64), np.asarray(R, dtype=np.float64)
    return [(float(q) * Q, float(r) * R) for q in q_scales for r in r_scales]


def select_noise(loglik, per: str = "fleet") -> Dict[str, np.ndarray]:
    """The maximum-likelihood choice from a host table ``loglik [C][n_tracks]`` of per-track scores.

    ``per="fleet"``: a track whose score is not finite under some candidate is excluded, so that every candidate is
    compared on the same tracks; the others are summed per candidate (``loglik [C]``) and ``best`` is one index.
    ``per="track"``: each track picks its own candidate (``best [n_tracks]``), a non-finite score counting as -inf;
    ``loglik`` is the table itself.  Ties go to the lowest candidate index.  ``excluded`` lists the tracks with a
    non-finite score under some candidate in either mode.  ``ValueError`` when the fleet comparison has no track left."""
    L = np.asarray(loglik.cpu().numpy() if hasattr(loglik, "cpu") else loglik, dtype=np.float64)
    if L.ndim != 2 or L.shape[0] < 1:
        raise ValueError(f"loglik must be a [C][n_tracks] table with C >= 1, got shape {L.shape}")
    finite = np.isfinite(L)
    excluded = np.flatnonzero(~finite.all(axis=0))
    if per == "fleet":
        keep = finite.all(axis=0)
        if not keep.any():
            raise ValueError("no track has a finite score under every candidate")
        sums = L[:, keep].sum(axis=1)
        return {"loglik": sums, "best": int(np.argmax(sums)), "excluded": excluded}
    if per == "track":
        best = np.argmax(np.where(finite, L, -np.inf), axis=0)   # argmax returns the first of equal maxima
        return {"loglik": L, "best": best.astype(np.int64), "excluded": excluded}
    raise ValueError(f"per must be 'fleet' or 'track', got {per!r}")


def fit_noise(engine, tiles, candidates: Sequence, per: str = "fleet") -> Dict[str, object]:
    """Score ``candidates`` (``(Q, R)`` pairs, e.g. :func:`noise_grid`) on every track of ``tiles`` with ``engine``
    (a ``BatchedUKF`` or ``BatchedUKFN``) and choose by maximum likelihood (:func:`select_noise`).

    ``tiles`` is one tile or a sequence of them, e.g. ``TrackBatchN.fleet_tiles`` output: column j of a tile is the
    caller's track ``tile.order[j]``; a tile without ``order`` holds the next ``n_tracks`` caller indices in sequence.
    Returns, in the caller's track order:
      ``loglik``   ``[C]`` fleet sums (``per="fleet"``) or the ``[C][n_tracks]`` table (``per="track"``);
      ``best``     the chosen candidate index, or one per track;
      ``Q``, ``R`` the chosen matrices, or one list entry per track (what ``TrackBatchN.from_tracks(Q=, R=)`` takes
                   at n = 5, and ``TrackBatch.from_tracks(Q=, R=)`` / ``TrackBatch.with_noise(Q=, R=)`` at n = 4, where a
                   per-track ``R`` selects the generic update);
      ``excluded`` the tracks with a non-finite score under some candidate (left out of the fleet sums).
    """
    tiles = [tiles] if hasattr(tiles, "n_tracks") else list(tiles)
    pairs = list(candidates)
    cols, parts, offset = [], [], 0
    for tile in tiles:
        T = tile.n_tracks
        cols.append(np.arange(offset, offset + T) if tile.order is None else np.asarray(tile.order, dtype=np.int64))
        offset += T
        parts.append(engine.score(tile, pairs)["loglik"])
    n_tracks = sum(len(c) for c in cols)
    table = np.full((len(pairs), n_tracks), np.nan)
    seen = np.zeros(n_tracks, dtype=bool)
    for c, part in zip(cols, parts):
        if len(c) and (c.min() < 0 or c.max() >= n_tracks):
            raise ValueError("the tiles' orders must cover each caller track exactly once")
        table[:, c] = part.cpu().numpy()
        seen[c] = True
    if not seen.all():   # as many columns as tracks: a track left out means another one twice
        raise ValueError("the tiles' orders must cover each caller track exactly once")
    pick = select_noise(table, per)
    if per == "fleet":
        Q, R = pairs[pick["best"]]
    else:
        Q, R = [pairs[k][0] for k in pick["best"]], [pairs[k][1] for k in pick["best"]]
    return {"loglik": pick["loglik"], "best": pick["best"], "Q": Q, "R": R, "excluded": pick["excluded"]}
