"""Fit metrics: the reference's three array helpers plus their whole-tile form on the device.

``rmse`` / ``cum_abs_diff`` / ``abs_diff`` keep the reference's names and meaning
(``performance_metrics.py:4-58``); they are array utilities on whatever the caller holds (numpy
arrays, or torch tensors on any device - the arithmetic then runs where the tensors live).
``track_metrics`` is what a 16 M-track run needs instead of copying every state to the host: one
kernel launch (``ste_track_metrics_f64``, ``ste_track_metrics_n_f64`` at n = 5) that reduces, per track, the residuals between a state
estimate and the observations it assimilated.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict

import numpy as np
import torch

from . import _native as nat

__all__ = ["rmse", "cum_abs_diff", "abs_diff", "track_metrics"]


def _is_tensor(*xs) -> bool:
    return any(isinstance(x, torch.Tensor) for x in xs)


def abs_diff(x, xref):
    """``|x - xref|`` element by element (performance_metrics.py:42-58)."""
    return (x - xref).abs() if _is_tensor(x, xref) else np.abs(x - xref)


def cum_abs_diff(x, xref):
    """Running sum of ``|x - xref|`` over the flattened arrays (performance_metrics.py:23-39)."""
    d = abs_diff(x, xref)
    return torch.cumsum(d.reshape(-1), 0) if _is_tensor(d) else np.cumsum(d)


def rmse(x, xref):
    """Root of the mean squared difference (performance_metrics.py:4-20)."""
    d = x - xref
    return torch.sqrt(torch.mean(d * d)) if _is_tensor(d) else np.sqrt(np.mean(d ** 2))


def track_metrics(ukf, batch, res, which: str = "smoothed", keep_abs_diff: bool = False) -> Dict[str, torch.Tensor]:
    """Per-track fit of a filtered (``which="filtered"``) or smoothed estimate to its observations.

    For every observation row the batch carries (longitude and latitude; speed and course too
    when the measurement model uses them) and every track: ``rmse``, the last element of
    ``cum_abs_diff`` and the maximum of ``abs_diff`` over the pairs (state after the update,
    observation), the prior being paired with the first fix.  Returns device tensors
    ``rmse``/``cum_abs``/``max_abs`` of shape ``[n, T]`` (NaN in rows the batch does not carry),
    ``n_pairs`` ``[T]`` and, on request, ``abs_diff`` ``[max_obs, n, T]``.

    ``n`` is 4 for a ``batch.BatchedUKF`` / ``TrackBatch`` / ``TrackResults`` triple
    (``ste_track_metrics_f64``) and 5 for a ``batch_n.BatchedUKFN`` / ``TrackBatchN`` / ``TrackResultsN``
    one (``ste_track_metrics_n_f64``); there the observations are the rows the forward pass
    assimilated, after the filter's measurement model.
    """
    from .batch_n import BatchedUKFN

    mean = {"smoothed": res.mean_s, "filtered": res.mean_f}[which]
    if mean is None:
        raise ValueError("results hold no smoothed states")
    ukf._check_shapes(batch, res, smoother=(which == "smoothed"))
    five = isinstance(ukf, BatchedUKFN)
    n, fn = (5, ukf._lib.ste_track_metrics_n_f64) if five else (4, ukf._lib.ste_track_metrics_f64)
    dev, T, ld = batch.device, batch.n_tracks, int(mean.shape[-1])
    out = {k: torch.full((n, ld), float("nan"), dtype=torch.float64, device=dev) for k in ("rmse", "cum_abs", "max_abs")}
    n_pairs = torch.zeros(ld, dtype=torch.int32, device=dev)
    ad = torch.full((batch.max_obs, n, ld), float("nan"), dtype=torch.float64, device=dev) if keep_abs_diff else None
    p, i = ukf._problem(batch), ukf._inputs(batch)
    with torch.cuda.device(dev):
        nat.check(fn(C.byref(p), C.byref(i), nat.ptr(mean), nat.ptr(out["rmse"]), nat.ptr(out["cum_abs"]), nat.ptr(out["max_abs"]),
                     nat.ptr(ad), nat.ptr(n_pairs), nat.current_stream()))
    out = {k: v[:, :T] for k, v in out.items()}
    out["n_pairs"] = n_pairs[:T]
    if ad is not None:
        out["abs_diff"] = ad[:, :, :T]
    return out
