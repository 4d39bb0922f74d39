"""Batched five-state UKF + URTSS over many tracks: the fleet path of ``geodetic_dynamics_turn``.

The state is ``[lon, lat, SOG, COG, COG rate]``, the turn rate a state that persists (the model behind
``UnscentedKalmanFilter(..., non_linear_process=geodetic_dynamics_turn)``).  :class:`TrackBatchN` is the
structure-of-arrays tile (track index fastest), :class:`BatchedUKFN` launches one whole-track forward
kernel and one ragged backward kernel per tile (``ste_ukf_forward_noise_n_f64`` /
``ste_urtss_backward_tracks_noise_n_f64``, with per-track ``Q`` / ``R`` when the tile has them) and
:class:`TrackResultsN` carries the per-step states back.

Every track is bit-identical to the dimension-generic single-step kernels driven step by step (the
class API's ``predict`` / ``update``) and to ``ste_urtss_backward_n_f64`` on that track alone: the
kernels share their arithmetic.  The host decisions - update mask, packing order, the smoother's rate
repeat and the ``IndexError`` rules - are those of :meth:`batch.TrackBatch.from_tracks`.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _native as nat
from .batch import (BatchedUKF, TrackBatch, TrackResults, copy_out, length_order, output_names, run_host_pipelined,
                    track_rate_repeat, track_rates, track_update_mask)

NS = 5   # state dimension of geodetic_dynamics_turn

#: default stored-state budget of a five-state tile (``sharding.plan_ragged_tiles``).  A stored state costs 480 B of
#: results (mean 5 + covariance 25 doubles, filtered and smoothed), and at most 65 B of inputs (dt and update flag per
#: step, five observation rows and two rates per fix; 120 B more with noise tapes).  The pipelined host path keeps two
#: input and two result sets resident, plus 80 B of diagonal scratch per state and set for ``outputs="cli"``:
#: 1e8 states take 2 x 48 GB + 2 x 6.5 GB (+ 24 GB with tapes) + 16 GB = 125 GB (149 GB) of a B200's 180 GB.
#: The n = 4 budget, 4e8 states, would need 384 GB for the two result sets alone.  Per-track ``Q`` / ``R`` add 400 B per
#: TRACK, not per state (25 doubles each, per input set): a tile of 1e8 states in 1e6 tracks carries 0.8 GB more.
STATE_BUDGET = 100_000_000


def _as55(name: str, M) -> np.ndarray:
    M = np.asarray(M, dtype=np.float64)
    if M.shape != (NS, NS):
        raise ValueError(f"{name} has shape {M.shape}: the five-state path takes 5 x 5 matrices")
    return np.ascontiguousarray(M)


def noise_planes(name: str, mats: Sequence, T: int) -> np.ndarray:
    """``[25][T]`` row-major planes of one symmetric 5 x 5 matrix per track (the layout of ``SteNoiseN.Q_tracks`` /
    ``R_tracks``); ``ValueError`` for a wrong count, shape or a non-symmetric matrix.  The kernels cannot check
    symmetry, so every per-track noise matrix passes through here."""
    if len(mats) != T:
        raise ValueError(f"{name}: {len(mats)} matrices for {T} tracks (one 5 x 5 matrix per track)")
    out = np.empty((NS * NS, T))
    for i, M in enumerate(mats):
        M = _as55(f"{name}[{i}]", M)
        if not np.array_equal(M, M.T):
            raise ValueError(f"{name}[{i}] must be symmetric")
        out[:, i] = M.reshape(-1)
    return out


@dataclass
class TrackBatchN:
    """Device-resident inputs of one tile of ``n_tracks`` five-state tracks (tensors ``[plane][track]``)."""

    x0: torch.Tensor  # [5][T]
    dt: torch.Tensor  # [max_steps][T]
    upd_mask: torch.Tensor  # [max_steps][T] uint8
    n_steps: torch.Tensor  # [T] int32
    sog_rate: torch.Tensor  # [max_obs][T]
    cog_rate: Optional[torch.Tensor]  # [max_obs][T]; the turn rate comes from the state, the kernels ignore it
    z: List[Optional[torch.Tensor]]  # 5 x [max_obs][T] (None = absent row, read as 0)
    rate_repeat: Optional[torch.Tensor] = None  # [T] int32, needed by the smoother
    P0: Optional[torch.Tensor] = None  # [25][T] per-track prior covariance
    noise_pred: Optional[torch.Tensor] = None  # [max_steps][5][T] unit normals
    noise_upd: Optional[torch.Tensor] = None  # [max_obs][5][T], row = update index
    noise_bwd: Optional[torch.Tensor] = None  # [max_steps][5][T], row = backward step
    # per-track noise, row-major 5 x 5 planes replacing the filter's shared matrix for each track (symmetric: from_tracks
    # and from_batch check it; check() cannot without a device synchronisation)
    Q: Optional[torch.Tensor] = None  # [25][T] process noise
    R: Optional[torch.Tensor] = None  # [25][T] measurement noise
    n_steps_host: Optional[np.ndarray] = None
    # column j holds the caller's track order[j] (ragged tiles are packed by decreasing length); None = caller's order
    order: Optional[np.ndarray] = None

    _TENSORS = ("x0", "dt", "upd_mask", "n_steps", "sog_rate", "cog_rate", "rate_repeat", "P0", "noise_pred", "noise_upd", "noise_bwd",
                "Q", "R")

    @property
    def n_tracks(self) -> int:
        return int(self.x0.shape[1])

    @property
    def max_steps(self) -> int:
        return int(self.dt.shape[0])

    @property
    def max_obs(self) -> int:
        return int(self.sog_rate.shape[0])

    @property
    def device(self) -> torch.device:
        return self.x0.device

    def track_steps(self) -> int:
        """Total filter steps in the tile (the unit of the throughput metric)."""
        if self.n_steps_host is not None:
            return int(self.n_steps_host.sum())
        return int(self.n_steps.sum().item())

    def check(self) -> None:
        """Shapes, dtypes, one device and contiguity of every tensor: the kernels trust them."""
        T, N, M, dev = self.n_tracks, self.max_steps, self.max_obs, self.device
        f64 = torch.float64
        expect = [("x0", self.x0, (NS, T), f64), ("dt", self.dt, (N, T), f64), ("upd_mask", self.upd_mask, (N, T), torch.uint8),
                  ("n_steps", self.n_steps, (T,), torch.int32), ("sog_rate", self.sog_rate, (M, T), f64),
                  ("cog_rate", self.cog_rate, (M, T), f64), ("rate_repeat", self.rate_repeat, (T,), torch.int32),
                  ("P0", self.P0, (NS * NS, T), f64), ("noise_pred", self.noise_pred, (N, NS, T), f64),
                  ("noise_upd", self.noise_upd, (M, NS, T), f64), ("noise_bwd", self.noise_bwd, (N, NS, T), f64),
                  ("Q", self.Q, (NS * NS, T), f64), ("R", self.R, (NS * NS, T), f64)]
        if len(self.z) != NS:
            raise ValueError("TrackBatchN.z must list the five observation rows (None for an absent row)")
        expect += [(f"z[{r}]", zr, (M, T), f64) for r, zr in enumerate(self.z)]
        for name, t, shape, dtype in expect:
            if t is None:
                if name in ("x0", "dt", "upd_mask", "n_steps", "sog_rate"):
                    raise ValueError(f"TrackBatchN.{name} is required")
                continue
            if tuple(t.shape) != shape or t.dtype != dtype or t.device != dev or not t.is_contiguous():
                raise ValueError(f"TrackBatchN.{name}: expected a contiguous {dtype} tensor of shape {shape} on {dev}, "
                                 f"got {t.dtype} {tuple(t.shape)} on {t.device}")
        if self.order is not None and len(self.order) != T:
            raise ValueError("TrackBatchN.order must have one entry per track")

    def _map(self, fn) -> "TrackBatchN":
        kw = {name: (None if getattr(self, name) is None else fn(getattr(self, name))) for name in self._TENSORS}
        return TrackBatchN(z=[None if r is None else fn(r) for r in self.z], n_steps_host=self.n_steps_host, order=self.order, **kw)

    def to(self, device, non_blocking: bool = False) -> "TrackBatchN":
        """Copy of the tile on ``device``."""
        return self._map(lambda t: t.to(device, non_blocking=non_blocking))

    def pin_memory(self) -> "TrackBatchN":
        """Host tile in page-locked memory (the staging form for :meth:`BatchedUKFN.run_host`)."""
        return self._map(lambda t: t.cpu().pin_memory())

    def copy_from(self, other: "TrackBatchN", non_blocking: bool = True) -> bool:
        """Overwrite this tile's tensors with ``other``'s (same shapes and the same optional tensors present; e.g.
        pinned host tile -> resident device tile, no allocation).  Returns False, with nothing copied, when the
        layouts differ."""
        pairs = [(getattr(self, n), getattr(other, n)) for n in self._TENSORS] + list(zip(self.z, other.z))
        if len(self.z) != len(other.z):
            return False
        for dst, src in pairs:
            if (dst is None) != (src is None) or (dst is not None and (dst.shape != src.shape or dst.dtype != src.dtype)):
                return False
        for dst, src in pairs:
            if dst is not None:
                dst.copy_(src, non_blocking=non_blocking)
        self.n_steps_host, self.order = other.n_steps_host, other.order
        if hasattr(self, "_z_model"):
            del self._z_model
        return True

    def input_bytes(self) -> int:
        """Bytes of every tensor of the tile (what one host->device upload moves)."""
        tensors = [getattr(self, n) for n in self._TENSORS] + list(self.z)
        return int(sum(t.numel() * t.element_size() for t in tensors if t is not None))

    @classmethod
    def fleet_tiles(cls, tracks: Sequence, dt_arrays: Sequence[np.ndarray], x0: Optional[Sequence[np.ndarray]] = None,
                    time0: float = 0.0, noise: Optional[Sequence[Optional[Dict[str, np.ndarray]]]] = None, smoother: bool = True,
                    device="cuda", P0: Optional[Sequence[np.ndarray]] = None, state_budget: Optional[int] = None,
                    Q: Optional[Sequence[np.ndarray]] = None, R: Optional[Sequence[np.ndarray]] = None, **plan) -> List["TrackBatchN"]:
        """A fleet too large for one tile, as tiles of :meth:`from_tracks` (same arguments): the tracks are sorted once
        by decreasing length and cut by ``sharding.plan_ragged_tiles`` (``state_budget`` stored states per tile,
        default :data:`STATE_BUDGET`; ``plan``: its ``granule`` / ``max_tracks``).  Column j of a tile holds the
        caller's track ``tile.order[j]``, and its results' ``track(i)`` takes that caller index."""
        from .sharding import plan_ragged_tiles

        if len(tracks) == 0:
            raise ValueError("empty batch")
        for name, mats in (("Q", Q), ("R", R)):
            if mats is not None:
                noise_planes(name, mats, len(tracks))   # errors name the caller's index, before any tile is built
        dt_arrays = [np.asarray(d, dtype=np.float64).reshape(-1) for d in dt_arrays]
        order = length_order([len(d) for d in dt_arrays])
        order = np.arange(len(tracks)) if order is None else order
        budget = STATE_BUDGET if state_budget is None else int(state_budget)
        tiles = []
        for lo, hi in plan_ragged_tiles([len(dt_arrays[j]) for j in order], budget, **plan):
            idx = order[lo:hi]
            pick = lambda seq: None if seq is None else [seq[j] for j in idx]   # noqa: E731
            tile = cls.from_tracks(pick(tracks), pick(dt_arrays), x0=pick(x0), time0=time0, noise=pick(noise), smoother=smoother,
                                   sort_by_length=False, device=device, P0=pick(P0), Q=pick(Q), R=pick(R))
            tile.order = np.array(idx)
            tiles.append(tile)
        return tiles

    # ------------------------------------------------------------------ #
    @classmethod
    def from_tracks(cls, tracks: Sequence, dt_arrays: Sequence[np.ndarray], x0: Optional[Sequence[np.ndarray]] = None,
                    time0: float = 0.0, noise: Optional[Sequence[Optional[Dict[str, np.ndarray]]]] = None, smoother: bool = True,
                    sort_by_length: bool = True, device="cuda", P0: Optional[Sequence[np.ndarray]] = None,
                    Q: Optional[Sequence[np.ndarray]] = None, R: Optional[Sequence[np.ndarray]] = None) -> "TrackBatchN":
        """Pack ``ShipTrack``-like objects (``dts, z, sog_rate, cog_rate``) with their step grids, as
        :meth:`TrackBatch.from_tracks` does.  ``z`` has 4 or 5 rows and is zero-padded to 5; the default
        ``x0`` is its padded first column.  ``noise``: per track ``None`` or a dict of unit normals
        ``pred (n_steps, 5)``, ``upd (n_updates, 5)``, ``bwd (n_steps, 5)`` (backward tape indexed by step).
        ``P0``: one 5 x 5 prior covariance per track instead of the filter's shared one (used as given, e.g. the
        not exactly symmetric covariance a previous run ended with).  ``Q`` / ``R``: one symmetric 5 x 5 process /
        measurement noise matrix per track, in the caller's order, instead of the filter's shared one (each track then
        equals a filter built with its own matrices; ``ValueError`` for a wrong count, shape or an asymmetric matrix).
        Raises ``IndexError`` where the reference would."""
        T = len(tracks)
        if T == 0:
            raise ValueError("empty batch")
        planes = {name: noise_planes(name, mats, T) for name, mats in (("Q", Q), ("R", R)) if mats is not None}
        dt_arrays = [np.asarray(d, dtype=np.float64).reshape(-1) for d in dt_arrays]
        order = length_order([len(d) for d in dt_arrays]) if sort_by_length else None
        if order is not None:
            tracks = [tracks[j] for j in order]
            dt_arrays = [dt_arrays[j] for j in order]
            x0 = None if x0 is None else [x0[j] for j in order]
            noise = None if noise is None else [noise[j] for j in order]
            P0 = None if P0 is None else [P0[j] for j in order]
            planes = {name: pl[:, order] for name, pl in planes.items()}
        nsteps = np.array([len(d) for d in dt_arrays], dtype=np.int32)
        nobs = np.array([np.asarray(tr.z).shape[1] for tr in tracks], dtype=np.int32)
        N, M = max(int(nsteps.max()), 1), int(nobs.max())
        dt, mask = np.zeros((N, T)), np.zeros((N, T), dtype=np.uint8)
        z, sr, cr = np.zeros((NS, M, T)), np.zeros((M, T)), np.zeros((M, T))
        x0a, rep = np.zeros((NS, T)), np.ones(T, dtype=np.int32)
        for i, tr in enumerate(tracks):
            zi = np.asarray(tr.z, dtype=np.float64)
            if zi.shape[0] not in (4, NS):
                raise ValueError(f"track {i}: z has {zi.shape[0]} rows; the five-state path takes 4 or 5")
            n, m = int(nsteps[i]), int(nobs[i])
            dt[:n, i] = dt_arrays[i]
            mask[:n, i] = track_update_mask(i, tr, dt_arrays[i], m, time0)
            z[: zi.shape[0], :m, i] = zi
            sr[:m, i], cr[:m, i] = track_rates(i, tr, m)
            x0a[:, i] = z[:, 0, i] if x0 is None else np.asarray(x0[i], dtype=np.float64).reshape(-1)
            if smoother:
                rep[i] = track_rate_repeat(i, tr, n, m)
        dev = torch.device(device)

        def up(a):
            return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

        kw = {name: up(pl) for name, pl in planes.items()}
        if P0 is not None:
            kw["P0"] = up(np.stack([_as55("P0", Pi) for Pi in P0], axis=-1).reshape(NS * NS, T))
        if noise is not None:
            npred, nupd, nbwd = np.zeros((N, NS, T)), np.zeros((M, NS, T)), np.zeros((N, NS, T))
            for i, nz in enumerate(noise):
                nz = nz or {}
                if nz.get("pred") is not None:
                    npred[: nsteps[i], :, i] = nz["pred"]
                if nz.get("upd") is not None:
                    nupd[: len(nz["upd"]), :, i] = nz["upd"]
                if nz.get("bwd") is not None:
                    nbwd[: nsteps[i], :, i] = nz["bwd"]
            kw.update(noise_pred=up(npred), noise_upd=up(nupd), noise_bwd=up(nbwd))
        return cls(x0=up(x0a), dt=up(dt), upd_mask=up(mask), n_steps=up(nsteps), sog_rate=up(sr), cog_rate=up(cr),
                   z=[up(z[r]) for r in range(NS)], rate_repeat=up(rep) if smoother else None, n_steps_host=nsteps.copy(),
                   order=order, **kw)

    @classmethod
    def from_batch(cls, b: TrackBatch, turn_rate0: float = 0.0, Q: Optional[Sequence[np.ndarray]] = None,
                   R: Optional[Sequence[np.ndarray]] = None) -> "TrackBatchN":
        """The five-state tile of an n = 4 tile already on the device (e.g. ``read_csv_fleet_device(...).to_batch()``):
        step grid, rates, observation rows, lengths and order are shared; the turn rate starts at ``turn_rate0``.  A
        tile in the cadence form (``upd_mask`` / ``n_steps`` / ``rate_repeat`` None) has them materialised on the
        device from ``substeps`` / ``rate_repeat_all``.  No host round trip.  ``Q`` / ``R``: one symmetric 5 x 5
        matrix per ship, in the caller's (ship) order, checked as by :meth:`from_tracks`; column j gets the matrix of
        ship ``b.order[j]``."""
        b.check()
        for name in ("P0", "R", "noise_pred", "noise_upd", "noise_bwd"):
            if getattr(b, name) is not None:
                raise ValueError(f"TrackBatch.{name} is 4-state data; build the five-state tile with TrackBatchN.from_tracks")
        dev, T, N = b.device, b.n_tracks, b.max_steps
        kw = {}
        for name, mats in (("Q", Q), ("R", R)):
            if mats is not None:
                pl = noise_planes(name, mats, T)
                kw[name] = torch.from_numpy(np.ascontiguousarray(pl if b.order is None else pl[:, b.order])).to(dev)
        x0 = torch.cat([b.x0, torch.full((1, T), float(turn_rate0), dtype=torch.float64, device=dev)]).contiguous()
        mask = b.upd_mask
        if mask is None:
            k = max(int(b.substeps), 1)
            every_k = ((torch.arange(N, device=dev) + 1) % k == 0).to(torch.uint8)
            mask = every_k[:, None].expand(N, T).contiguous()
        n_steps = b.n_steps if b.n_steps is not None else torch.full((T,), N, dtype=torch.int32, device=dev)
        rep = b.rate_repeat if b.rate_repeat is not None else torch.full((T,), max(int(b.rate_repeat_all), 1), dtype=torch.int32, device=dev)
        return cls(x0=x0, dt=b.dt, upd_mask=mask, n_steps=n_steps, sog_rate=b.sog_rate, cog_rate=b.cog_rate, z=list(b.z) + [None],
                   rate_repeat=rep, n_steps_host=b.n_steps_host, order=b.order, **kw)


@dataclass
class TrackResultsN:
    """Per-step states of a five-state tile: ``mean [N+1][5][T]``, ``cov [N+1][25][T]``."""

    mean_f: torch.Tensor
    cov_f: torch.Tensor
    mean_s: Optional[torch.Tensor]
    cov_s: Optional[torch.Tensor]
    status: torch.Tensor
    n_updates: torch.Tensor
    n_steps_host: Optional[np.ndarray] = None
    order: Optional[np.ndarray] = None
    filtered_by: Optional[int] = field(default=None, repr=False, compare=False)   # id() of the tile last filtered here
    _column_of: Optional[np.ndarray] = field(default=None, repr=False, compare=False)

    _TENSORS = ("mean_f", "cov_f", "mean_s", "cov_s", "status", "n_updates")

    def host_like(self, pinned: bool = True) -> "TrackResultsN":
        """Empty host buffers of the same shapes (page-locked by default) for device->host copies."""
        def mk(t):
            if t is None:
                return None
            h = torch.empty(t.shape, dtype=t.dtype, device="cpu")
            return h.pin_memory() if pinned else h
        return TrackResultsN(n_steps_host=self.n_steps_host, order=self.order, **{n: mk(getattr(self, n)) for n in self._TENSORS})

    def copy_to(self, other: "TrackResultsN", non_blocking: bool = True) -> int:
        """Copy every buffer into ``other`` (e.g. device -> pinned host); returns the bytes moved."""
        moved = 0
        for n in self._TENSORS:
            src, dst = getattr(self, n), getattr(other, n)
            if src is None or dst is None:
                continue
            dst.copy_(src, non_blocking=non_blocking)
            moved += src.numel() * src.element_size()
        return moved

    def to_host(self, pinned: bool = False) -> "TrackResultsN":
        """Host copy of every buffer (one device->host transfer per array); ``track(i)`` on it costs no further
        transfers - the form the fleet writers use."""
        if not self.mean_f.is_cuda:
            return self
        host = self.host_like(pinned=pinned)
        self.copy_to(host, non_blocking=pinned)
        if pinned:
            torch.cuda.current_stream(self.mean_f.device).synchronize()
        return host

    def check_status(self, raise_on: int = nat.STE_STATUS_NONFINITE | nat.STE_STATUS_OBS_OVERRUN) -> Dict[str, int]:
        """Per-track status bits as counts; raises ``IndexError`` for an observation overrun and
        ``FloatingPointError`` for non-finite states unless masked out of ``raise_on``."""
        return TrackResults.check_status(self, raise_on)   # reads only .status

    def column(self, i: int) -> int:
        """Column of the caller's track ``i`` (a tile of :meth:`TrackBatchN.fleet_tiles` holds some of the caller's
        tracks: ``IndexError`` for one it does not hold)."""
        if self.order is None:
            return int(i)
        if self._column_of is None:
            self._column_of = np.full(int(np.max(self.order)) + 1 if len(self.order) else 0, -1, dtype=np.int64)
            self._column_of[self.order] = np.arange(len(self.order))
        j = int(self._column_of[i]) if 0 <= i < len(self._column_of) else -1
        if j < 0:
            raise IndexError(f"track {i} is not in this tile")
        return j

    def track(self, i: int) -> Dict[str, np.ndarray]:
        """Host copies for the caller's track ``i``: means (N_i+1, 5), covs (N_i+1, 5, 5)[, means_s, covs_s]."""
        j = self.column(i)
        n = int(self.n_steps_host[j]) if self.n_steps_host is not None else self.mean_f.shape[0] - 1
        out = {"means": self.mean_f[: n + 1, :, j].cpu().numpy(),
               "covs": self.cov_f[: n + 1, :, j].cpu().numpy().reshape(n + 1, NS, NS),
               "status": int(self.status[j].item()), "n_updates": int(self.n_updates[j].item())}
        if self.mean_s is not None:
            out["means_s"] = self.mean_s[: n + 1, :, j].cpu().numpy()
            out["covs_s"] = self.cov_s[: n + 1, :, j].cpu().numpy().reshape(n + 1, NS, NS)
        return out


class BatchedUKFN:
    """Five-state UKF forward filter + URTSS backward smoother over a :class:`TrackBatchN` on one GPU.

    Results parity contract: every track equals the class API's ``run`` / ``run_rts_smoother`` at n = 5 on
    the same inputs (bit for bit), with the noise draws zero or replayed from the tile's tapes."""

    def __init__(self, H, Q=None, R=None, P=None, process=None, measurement_model=None, *, gating=False):
        from .kalman_filters.non_linear_process import DEVICE_MODELS, geodetic_dynamics, geodetic_dynamics_turn
        from .measurement_models import MEASUREMENT_MODELS

        if H is None:
            raise ValueError("Set proper system dynamics.")
        process = geodetic_dynamics_turn if process is None else process
        if process is geodetic_dynamics:
            raise ValueError("geodetic_dynamics is the n = 4 model: use batch.BatchedUKF")
        if DEVICE_MODELS.get(process) != (nat.STE_MODEL_GEODETIC_TURN, NS):
            raise NotImplementedError("BatchedUKFN runs geodetic_dynamics_turn (n = 5)")
        if gating:
            raise NotImplementedError("the robustification is implemented for the n = 4 state (BatchedUKF)")
        if measurement_model is not None and measurement_model not in MEASUREMENT_MODELS.values():
            raise NotImplementedError("measurement_model must be one of ship_track_estimators_b200.measurement_models."
                                      f"{sorted(MEASUREMENT_MODELS)} (arbitrary callables cannot run inside the kernels)")
        eye = np.eye(NS)
        self.H = _as55("H", H)
        self.Q = _as55("Q", eye if Q is None else Q)
        self.R = _as55("R", eye if R is None else R)
        self.P0 = _as55("P", eye if P is None else P)
        for name in ("Q", "R", "P0"):
            M = getattr(self, name)
            if not np.array_equal(M, M.T):
                raise ValueError(f"{name} must be symmetric")
        self.measurement_model = measurement_model
        self._lib = nat.load()
        self._pipe = None   # streams and resident buffers of run_host_pipelined, created once

    def _problem(self, b: TrackBatchN) -> nat.SteProblemN:
        p = nat.SteProblemN()
        p.n, p.model, p.n_tracks, p.max_steps, p.max_obs, p.ld = NS, nat.STE_MODEL_GEODETIC_TURN, b.n_tracks, b.max_steps, b.max_obs, b.n_tracks
        for name, M in (("H", self.H), ("Q", self.Q), ("R", self.R), ("P0", self.P0)):
            getattr(p, name)[: NS * NS] = M.reshape(-1).tolist()
        return p

    def _rows(self, b: TrackBatchN):
        if self.measurement_model is None:
            return b.z
        cached = getattr(b, "_z_model", None)
        if cached is None or cached[0] is not self.measurement_model:
            from .measurement_models import apply_rows, position_only

            rows = apply_rows(self.measurement_model, b.z[:4])
            rows.append(None if self.measurement_model is position_only else b.z[4])   # the element-wise models keep 0 at 0
            cached = b._z_model = (self.measurement_model, rows)
        return cached[1]

    def _inputs(self, b: TrackBatchN) -> nat.SteInputsN:
        i = nat.SteInputsN()
        i.x0, i.P0, i.dt, i.upd_mask, i.n_steps = (nat.ptr(getattr(b, n)) for n in ("x0", "P0", "dt", "upd_mask", "n_steps"))
        for r, zr in enumerate(self._rows(b)):
            i.z[r] = nat.ptr(zr)
        i.sog_rate, i.cog_rate, i.rate_repeat = nat.ptr(b.sog_rate), nat.ptr(b.cog_rate), nat.ptr(b.rate_repeat)
        i.noise_pred, i.noise_upd, i.noise_bwd = nat.ptr(b.noise_pred), nat.ptr(b.noise_upd), nat.ptr(b.noise_bwd)
        return i

    @staticmethod
    def _noise(b: TrackBatchN) -> nat.SteNoiseN:
        return nat.SteNoiseN(nat.ptr(b.Q), nat.ptr(b.R))

    @staticmethod
    def _outputs(r: TrackResultsN) -> nat.SteOutputsN:
        o = nat.SteOutputsN()
        o.mean_f, o.cov_f, o.mean_s, o.cov_s = nat.ptr(r.mean_f), nat.ptr(r.cov_f), nat.ptr(r.mean_s), nat.ptr(r.cov_s)
        o.status, o.n_updates = nat.ptr(r.status), nat.ptr(r.n_updates)
        return o

    def allocate(self, b: TrackBatchN, smoother: bool = True) -> TrackResultsN:
        """Output buffers for a tile (reusable across tiles of the same shape)."""
        dev, T, S = b.device, b.n_tracks, b.max_steps + 1
        f64 = dict(dtype=torch.float64, device=dev)
        return TrackResultsN(
            mean_f=torch.empty(S, NS, T, **f64), cov_f=torch.empty(S, NS * NS, T, **f64),
            mean_s=torch.empty(S, NS, T, **f64) if smoother else None, cov_s=torch.empty(S, NS * NS, T, **f64) if smoother else None,
            status=torch.zeros(T, dtype=torch.int32, device=dev), n_updates=torch.zeros(T, dtype=torch.int32, device=dev),
            n_steps_host=b.n_steps_host, order=b.order)

    def _check_shapes(self, b: TrackBatchN, res: TrackResultsN, smoother: bool = False) -> None:
        b.check()
        T, S, dev = b.n_tracks, b.max_steps + 1, b.device
        expect = [("mean_f", res.mean_f, (S, NS, T)), ("cov_f", res.cov_f, (S, NS * NS, T)), ("status", res.status, (T,)),
                  ("n_updates", res.n_updates, (T,))]
        if smoother:
            if res.mean_s is None or res.cov_s is None:
                raise ValueError("results were allocated without smoother buffers")
            expect += [("mean_s", res.mean_s, (S, NS, T)), ("cov_s", res.cov_s, (S, NS * NS, T))]
        for name, t, shape in expect:
            if t is None or tuple(t.shape) != shape or t.device != dev or not t.is_contiguous():
                got = "None" if t is None else f"{tuple(t.shape)} on {t.device}"
                raise ValueError(f"TrackResultsN.{name}: expected a contiguous tensor of shape {shape} on {dev} for this tile, got {got}")

    def forward(self, b: TrackBatchN, res: TrackResultsN) -> None:
        """Launch the forward filter (asynchronous on the current stream)."""
        self._check_shapes(b, res)
        p, i, o = self._problem(b), self._inputs(b), self._outputs(res)
        res.filtered_by = id(b)
        with torch.cuda.device(b.device):
            nat.check(self._lib.ste_ukf_forward_noise_n_f64(C.byref(p), C.byref(i), C.byref(self._noise(b)), C.byref(o),
                                                            nat.current_stream()))

    def backward(self, b: TrackBatchN, res: TrackResultsN) -> None:
        """Launch the URTSS backward pass over the filtered states in ``res`` (written by ``forward(b, res)``)."""
        self._check_shapes(b, res, smoother=True)
        if res.filtered_by is not None and res.filtered_by != id(b):
            raise ValueError("these results were last filtered from a different tile: run forward() on this tile first")
        if b.rate_repeat is None:
            raise ValueError("the smoother needs TrackBatchN.rate_repeat (from_tracks(..., smoother=True))")
        p, i, o = self._problem(b), self._inputs(b), self._outputs(res)
        with torch.cuda.device(b.device):
            nat.check(self._lib.ste_urtss_backward_tracks_noise_n_f64(C.byref(p), C.byref(i), C.byref(self._noise(b)), C.byref(o),
                                                                      nat.current_stream()))

    def run(self, b: TrackBatchN, smoother: bool = True, res: Optional[TrackResultsN] = None) -> TrackResultsN:
        res = res if res is not None else self.allocate(b, smoother=smoother)
        self.forward(b, res)
        if smoother:
            self.backward(b, res)
        return res

    def run_many(self, batches: Sequence[TrackBatchN], results: Sequence[TrackResultsN]) -> None:
        """Filter and smooth a sequence of resident tiles (e.g. :meth:`TrackBatchN.fleet_tiles`): two launches per tile,
        on the current stream."""
        if len(batches) != len(results):
            raise ValueError("one result set per tile")
        for b, r in zip(batches, results):
            self.forward(b, r)
            self.backward(b, r)

    # ------------------------------------------------------------------ #
    # host-buffer (end-to-end) entry points, as BatchedUKF's              #
    # ------------------------------------------------------------------ #
    #: named selections of what travels back to the host per tile (the names of ``BatchedUKF.OUTPUT_SETS``).  Per
    #: stored state: "all" 480 B, "cli" 160 B (means and diag(P) of both passes, what the CLI writes), "filtered" and
    #: "smoothed" 80 B each, "summary" nothing per state: per track the last filtered state (5 + 25) and the fit
    #: metrics of ``performance_metrics.track_metrics`` (3 x 5).
    OUTPUT_SETS = BatchedUKF.OUTPUT_SETS
    _DIAG = [r * NS + r for r in range(NS)]   # planes 0, 6, 12, 18, 24

    def _output_names(self, outputs, smoother: bool):
        return output_names(self.OUTPUT_SETS, outputs, smoother)

    def host_outputs(self, b: TrackBatchN, outputs="all", smoother: bool = True, pinned: bool = True) -> Dict[str, torch.Tensor]:
        """Host buffers (page-locked by default) for the selected outputs of a tile shaped like ``b``, plus the
        always-returned per-track ``status`` and ``n_updates``."""
        T, S = b.n_tracks, b.max_steps + 1
        shapes = {"mean_f": (S, NS, T), "mean_s": (S, NS, T), "cov_f": (S, NS * NS, T), "cov_s": (S, NS * NS, T),
                  "diag_f": (S, NS, T), "diag_s": (S, NS, T), "final": (NS + NS * NS, T), "metrics": (3 * NS, T)}
        out = {}
        for n in self._output_names(outputs, smoother) + ("status", "n_updates"):
            t = torch.empty(shapes.get(n, (T,)), dtype=torch.int32 if n in ("status", "n_updates") else torch.float64)
            out[n] = t.pin_memory() if pinned else t
        return out

    def _extract(self, b: TrackBatchN, res: TrackResultsN, names, smoother: bool, scratch: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """Device tensors for the selected outputs (views where the result buffers already hold them, small gathers
        into ``scratch`` otherwise)."""
        dev = b.device
        dsel = scratch.get("_diag_idx")
        if dsel is None:
            dsel = scratch["_diag_idx"] = torch.tensor(self._DIAG, device=dev)
        out = {"status": res.status, "n_updates": res.n_updates}
        for n in names:
            if n in ("mean_f", "cov_f", "mean_s", "cov_s"):
                out[n] = getattr(res, n)
            elif n in ("diag_f", "diag_s"):
                cov = res.cov_f if n == "diag_f" else res.cov_s
                buf = scratch.get(n)
                if buf is None or buf.shape != (cov.shape[0], NS, cov.shape[2]):
                    buf = scratch[n] = torch.empty(cov.shape[0], NS, cov.shape[2], dtype=torch.float64, device=dev)
                torch.index_select(cov, 1, dsel, out=buf)
                out[n] = buf
            elif n == "final":
                last = b.n_steps.to(torch.int64)[None, None, :]
                out[n] = torch.cat([torch.gather(res.mean_f, 0, last.expand(1, NS, -1))[0],
                                    torch.gather(res.cov_f, 0, last.expand(1, NS * NS, -1))[0]], dim=0)
            elif n == "metrics":
                from .performance_metrics import track_metrics

                m = track_metrics(self, b, res, which="smoothed" if smoother else "filtered")
                out[n] = torch.cat([m["rmse"], m["cum_abs"], m["max_abs"]], dim=0)
        return out

    def run_host(self, host_batch: TrackBatchN, host_out, dev_res: Optional[TrackResultsN] = None, smoother: bool = True,
                 device="cuda", outputs="all") -> Dict[str, int]:
        """End-to-end call on HOST buffers: pinned inputs -> device, forward (+ backward), the selected ``outputs`` ->
        pinned ``host_out`` (a dict from :meth:`host_outputs`, or a host ``TrackResultsN`` for ``outputs="all"``).
        Asynchronous on the current stream; synchronise before reading ``host_out``.  Returns the bytes copied in
        each direction."""
        names = self._output_names(outputs, smoother)
        dev_batch = host_batch.to(device, non_blocking=True)
        dev_res = self.run(dev_batch, smoother=smoother, res=dev_res)
        d2h = copy_out(self._extract(dev_batch, dev_res, names, smoother, {}), host_out)
        return {"h2d_bytes": host_batch.input_bytes(), "d2h_bytes": d2h}

    def run_host_pipelined(self, host_batches: Sequence[TrackBatchN], host_outs: Sequence, smoother: bool = True,
                           device="cuda", outputs="all") -> Dict[str, int]:
        """:meth:`BatchedUKF.run_host_pipelined` for five-state tiles: while tile i is filtered and smoothed, tile
        i+1's inputs travel host->device and tile i-1's selected ``outputs`` device->host, on three streams with two
        resident buffer sets.  ``host_batches`` / ``host_outs`` live in pinned memory and all tiles share one shape
        (``ValueError`` otherwise).  Returns the bytes copied over all tiles in each direction; synchronise before
        reading ``host_outs``."""
        return run_host_pipelined(self, host_batches, host_outs, self._output_names(outputs, smoother), smoother, device)
