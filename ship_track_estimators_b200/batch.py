"""Batched UKF + URTSS over many independent tracks: the B200-native entry point.

The reference has no batched API ("batch" there is a Python loop over ships,
``examples/example_ukf_rts_smoother_batch.py:19``); this module is what that loop becomes.  A
:class:`TrackBatch` is the structure-of-arrays tile the kernels read (track index fastest),
:class:`BatchedUKF` launches the forward filter and the backward smoother through the C ABI and
:class:`TrackResults` carries the per-step states back.  The single-track
``UnscentedKalmanFilter`` class of the reference API is a batch of one on top of this.

Host-side decisions that must match the reference exactly are taken here, once per track, with
the reference's own arithmetic (numpy fp64):
  * which steps assimilate an observation: ``self.time += dt`` against ``np.cumsum(dts)`` by exact
    float equality (reference ``kalman_filter.py:73, 98, 101``) -> ``upd_mask``;
  * the smoother's rate expansion ``np.repeat(rate, int(nstates / len(dts)))`` (reference
    ``unscented.py:287-292``) -> ``rate_repeat``.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field, replace
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _native as nat


def _as44(name: str, M) -> np.ndarray:
    M = np.asarray(M, dtype=np.float64)
    if M.shape != (4, 4):
        raise NotImplementedError(
            f"{name} has shape {M.shape}: the CUDA UKF path is built for the n = 4 state "
            "[lon, lat, SOG, COG] (the reference's update/rts_step hard-code state index 3 as heading)"
        )
    return np.ascontiguousarray(M)


def track_planes(name: str, mats: Sequence, T: int) -> np.ndarray:
    """``[16][T]`` row-major planes of one symmetric 4 x 4 matrix per track (the layout of ``SteInputs.R_tracks`` and
    ``SteNoiseN.Q_tracks``), column ``i`` from ``mats[i]``.  ``ValueError`` for a wrong count; a wrong shape or an asymmetric
    matrix raises as ``from_tracks(R=)`` does.  The kernels cannot check symmetry, so per-track matrices pass through here."""
    if len(mats) != T:
        raise ValueError(f"{name}: {len(mats)} matrices for {T} tracks (one 4 x 4 matrix per track)")
    out = np.empty((16, T))
    for i, M in enumerate(mats):
        M = _as44(f"{name}[{i}]", M)
        if not np.array_equal(M, M.T):
            raise NotImplementedError(f"per-track {name} must be symmetric for the CUDA path ({name}[{i}] is not)")
        out[:, i] = M.reshape(-1)
    return out


@dataclass
class FilterModel:
    """H, Q, R, P0 of ``UnscentedKalmanFilter.__init__`` (reference ``unscented.py:20-74``) plus the
    robustification switch (reference ``unscented.py:353-387``, disabled there)."""

    H: np.ndarray
    Q: np.ndarray
    R: np.ndarray
    P0: np.ndarray
    gating: bool = False
    gate_chi: float = 50.0
    gate_max_iter: int = 100
    force_generic: bool = False

    def __post_init__(self):
        self.H = _as44("H", self.H)
        self.Q = _as44("Q", self.Q)
        self.R = _as44("R", self.R)
        self.P0 = _as44("P", self.P0)
        for name in ("Q", "R", "P0"):
            M = getattr(self, name)
            if not np.array_equal(M, M.T):
                raise NotImplementedError(f"{name} must be symmetric for the CUDA path")

    def position_only(self) -> bool:
        """Whether the kernels take the position-only update: H = diag(1,1,0,0) exactly, R zero outside its
        leading 2x2 block and no ``force_generic``."""
        return (not self.force_generic) and np.array_equal(self.H, np.diag([1.0, 1.0, 0.0, 0.0])) and not (
            np.any(self.R[2:, :]) or np.any(self.R[:, 2:])
        )

    def rows_needed(self) -> List[bool]:
        """Observation rows the update can actually read (a row multiplying only exact zeros of
        pinv(H P H^T + R) may be absent)."""
        if self.position_only():
            return [True, True, False, False]
        return [bool(self.gating or np.any(self.H[r]) or np.any(self.R[r])) for r in range(4)]


def exact_update_mask(dt_array: np.ndarray, dts: np.ndarray, time0: float = 0.0) -> np.ndarray:
    """Steps whose accumulated time equals an observation time exactly.

    ``self.time += dt`` (reference ``kalman_filter.py:98``) and ``np.cumsum`` (``:73``) are both
    sequential fp64 sums; ``in`` (``:101``) is float equality against any element.
    """
    dt_array = np.asarray(dt_array, dtype=np.float64)
    if dt_array.size == 0:
        return np.zeros(0, dtype=bool)
    if time0 == 0:
        times = np.cumsum(dt_array)
    else:
        times = np.cumsum(np.concatenate(([np.float64(time0)], dt_array)))[1:]
    return np.isin(times, np.cumsum(np.asarray(dts, dtype=np.float64)))


def length_order(lengths) -> Optional[np.ndarray]:
    """Packing order of a ragged fleet: decreasing length, stable (equal lengths keep the caller's
    order); None when the tracks are already in that order."""
    lengths = np.asarray(lengths)
    if len(lengths) > 1 and np.any(lengths[:-1] < lengths[1:]):
        return np.argsort(-lengths, kind="stable")
    return None


def track_update_mask(i: int, tr, dt_array: np.ndarray, m: int, time0: float = 0.0) -> np.ndarray:
    """``exact_update_mask`` of track ``i`` with ``m`` observations; ``IndexError`` where the reference
    raises it: more matched observation times than observations (``kalman_filter.py:101-108``)."""
    mk = exact_update_mask(dt_array, tr.dts, time0)
    if 1 + int(mk.sum()) > m:
        raise IndexError(f"track {i}: {1 + int(mk.sum())} update times matched but only {m} observations")
    return mk


def track_rates(i: int, tr, m: int):
    """The first ``m`` entries of the track's ``sog_rate`` / ``cog_rate`` (``IndexError`` if shorter)."""
    sri, cri = np.asarray(tr.sog_rate, dtype=np.float64), np.asarray(tr.cog_rate, dtype=np.float64)
    if len(sri) < m or len(cri) < m:
        raise IndexError(f"track {i}: sog_rate/cog_rate shorter than the observations")
    return sri[:m], cri[:m]


def track_rate_repeat(i: int, tr, n: int, m: int) -> int:
    """The smoother's ``int(nstates / len(dts))`` rate repeat of a track of ``n`` steps and ``m``
    observations (reference ``unscented.py:287-292``); ``IndexError`` when a rate index runs past the
    repeated arrays (``:287-311``)."""
    r = int((n + 1) / max(len(np.asarray(tr.dts)), 1)) if len(np.asarray(tr.dts)) else 0
    if r < 1 or (n > 0 and (n - 1) // r >= m):
        raise IndexError(f"track {i}: smoother rate index out of range (repeat {r})")
    return r


@dataclass
class TrackBatch:
    """Device-resident inputs of one tile of ``n_tracks`` tracks (all tensors ``[plane][track]``)."""

    x0: torch.Tensor  # [4][T]
    dt: torch.Tensor  # [max_steps][T]
    sog_rate: torch.Tensor  # [max_obs][T]
    cog_rate: torch.Tensor  # [max_obs][T]
    z: List[Optional[torch.Tensor]]  # 4 x [max_obs][T] (rows lon, lat, sog, cog)
    upd_mask: Optional[torch.Tensor] = None  # [max_steps][T] uint8; None -> every `substeps`-th step
    n_steps: Optional[torch.Tensor] = None  # [T] int32; None -> max_steps for all
    rate_repeat: Optional[torch.Tensor] = None  # [T] int32; None -> rate_repeat_all
    substeps: int = 1
    rate_repeat_all: int = 1
    P0: Optional[torch.Tensor] = None  # [16][T] per-track prior covariance
    R: Optional[torch.Tensor] = None  # [16][T] per-track measurement covariance (ships with different sensors)
    noise_pred: Optional[torch.Tensor] = None  # [max_steps][4][T] unit normals
    noise_upd: Optional[torch.Tensor] = None  # [max_obs][4][T]
    noise_bwd: Optional[torch.Tensor] = None  # [max_steps][4][T]
    n_steps_host: Optional[np.ndarray] = None  # host copy for result slicing
    # ragged tiles are packed in order of decreasing length (warps retire together, freed block slots
    # take the next longest tracks): column j holds the caller's track order[j]; None = caller's order
    order: Optional[np.ndarray] = None
    _long_fraction: Optional[float] = field(default=None, repr=False, compare=False)
    # per-track process noise (fleets mixing ship classes): row-major 4 x 4 planes replacing the filter's shared Q for
    # each track in both passes (symmetric: from_tracks and with_noise check it; check() cannot without a synchronisation)
    Q: Optional[torch.Tensor] = None  # [16][T]

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
        if self.n_steps is not None:
            return int(self.n_steps.sum().item())
        return self.n_tracks * self.max_steps

    def check(self) -> None:
        """Consistency of the tile's own tensors (row counts, track count, dtypes, one device); the
        kernels trust these shapes, so a mismatch would read or write out of bounds."""
        T, N, M, dev = self.n_tracks, self.max_steps, self.max_obs, self.device
        f64, expect = torch.float64, []
        expect += [("x0", self.x0, (4, T), f64), ("dt", self.dt, (N, T), f64), ("sog_rate", self.sog_rate, (M, T), f64),
                   ("cog_rate", self.cog_rate, (M, T), f64), ("upd_mask", self.upd_mask, (N, T), torch.uint8),
                   ("n_steps", self.n_steps, (T,), torch.int32), ("rate_repeat", self.rate_repeat, (T,), torch.int32),
                   ("P0", self.P0, (16, T), f64), ("R", self.R, (16, T), f64), ("noise_pred", self.noise_pred, (N, 4, T), f64),
                   ("noise_upd", self.noise_upd, (M, 4, T), f64), ("noise_bwd", self.noise_bwd, (N, 4, T), f64),
                   ("Q", self.Q, (16, T), f64)]
        expect += [(f"z[{r}]", zr, (M, T), f64) for r, zr in enumerate(self.z)]
        for name, t, shape, dtype in expect:
            if t is None:
                continue
            if tuple(t.shape) != shape or t.dtype != dtype or t.device != dev or not t.is_contiguous():
                raise ValueError(f"TrackBatch.{name}: expected a contiguous {dtype} tensor of shape {shape} on {dev}, "
                                 f"got {t.dtype} {tuple(t.shape)} on {t.device}")
        if len(self.z) != 4:
            raise ValueError("TrackBatch.z must list the four observation rows (None for an absent row)")
        if self.order is not None and len(self.order) != T:
            raise ValueError("TrackBatch.order must have one entry per track")

    def long_step_fraction(self, limit_km: float = 90.0) -> float:
        """Fraction of the tile's legs (fix to next fix, divided over the sub-steps) longer than
        ``limit_km`` - a little inside the 100 km range of the geodetic step's small-displacement tier.
        A value well between 0 and 1 means the lanes of a warp would split between the two tiers;
        ``BatchedUKF`` then keeps the tile on the full-range tier (``STE_FLAG_LONG_STEPS``).  Computed
        once per tile (one device reduction) and cached."""
        if self._long_fraction is None:
            self._long_fraction = self._long_step_fraction(limit_km)
        return self._long_fraction

    def _long_step_fraction(self, limit_km: float) -> float:
        lon, lat = self.z[0], self.z[1]
        if lon is None or lat is None or lon.shape[0] < 2:
            return 0.0
        rad = torch.pi / 180.0
        p1, p2, dl = lat[:-1] * rad, lat[1:] * rad, (lon[1:] - lon[:-1]) * rad
        a = torch.sin((p2 - p1) / 2) ** 2 + torch.cos(p1) * torch.cos(p2) * torch.sin(dl / 2) ** 2
        km = 2.0 * 6371.0 * torch.asin(torch.sqrt(a.clamp(0.0, 1.0))) / max(int(self.substeps), 1)
        legs = torch.arange(lon.shape[0] - 1, device=lon.device)[:, None]
        if self.n_steps is not None:     # legs a track really has: n_steps / substeps (from_tracks stores substeps = 1)
            n_legs = (self.n_steps.to(torch.int64) // max(int(self.substeps), 1)).clamp(max=lon.shape[0] - 1)
            valid = legs < n_legs[None, :]
        else:
            valid = torch.ones_like(km, dtype=torch.bool)
        total = int(valid.sum())
        return float(((km > limit_km) & valid).sum()) / total if total else 0.0

    _TENSORS = ("x0", "dt", "sog_rate", "cog_rate", "upd_mask", "n_steps", "rate_repeat", "P0", "R",
                "noise_pred", "noise_upd", "noise_bwd", "Q")

    def _map(self, fn) -> "TrackBatch":
        kw = {name: (None if getattr(self, name) is None else fn(getattr(self, name))) for name in self._TENSORS}
        return TrackBatch(z=[None if r is None else fn(r) for r in self.z], substeps=self.substeps,
                          rate_repeat_all=self.rate_repeat_all, n_steps_host=self.n_steps_host, order=self.order,
                          _long_fraction=self._long_fraction, **kw)

    def to(self, device, non_blocking: bool = False) -> "TrackBatch":
        """Copy of the tile on ``device`` (host->device copies are asynchronous from pinned memory)."""
        return self._map(lambda t: t.to(device, non_blocking=non_blocking))

    def copy_from(self, other: "TrackBatch", non_blocking: bool = True) -> bool:
        """Overwrite this tile's tensors with ``other``'s (same shapes and the same optional tensors
        present; e.g. pinned host tile -> resident device tile, no allocation).  Returns False, with
        nothing copied, when the layouts differ."""
        pairs = [(getattr(self, n), getattr(other, n)) for n in self._TENSORS] + list(zip(self.z, other.z))
        for dst, src in pairs:
            if (dst is None) != (src is None) or (dst is not None and (dst.shape != src.shape or dst.dtype != src.dtype)):
                return False
        for dst, src in pairs:
            if dst is not None:
                dst.copy_(src, non_blocking=non_blocking)
        self.substeps, self.rate_repeat_all = other.substeps, other.rate_repeat_all
        self.n_steps_host, self.order, self._long_fraction = other.n_steps_host, other.order, other._long_fraction
        if hasattr(self, "_z_model"):
            del self._z_model
        return True

    def pin_memory(self) -> "TrackBatch":
        """Host tile in page-locked memory (the staging form for :meth:`BatchedUKF.run_host`)."""
        return self._map(lambda t: t.cpu().pin_memory())

    def input_bytes(self) -> int:
        total = sum(r.numel() * r.element_size() for r in self.z if r is not None)
        for name in self._TENSORS:
            t = getattr(self, name)
            total += 0 if t is None else t.numel() * t.element_size()
        return int(total)

    def with_noise(self, Q: Optional[Sequence[np.ndarray]] = None, R: Optional[Sequence[np.ndarray]] = None) -> "TrackBatch":
        """This tile with per-track noise: ``Q`` / ``R`` give one symmetric 4 x 4 matrix per ship in the caller's (ship)
        order, checked as by :meth:`from_tracks`, and column j gets the matrix of ship ``order[j]``.  A set that is given
        replaces the tile's own, one that is not keeps it; every other tensor is shared.  For tiles built on the device
        (``FleetFixes.to_batch``, ``read_csv_fleet_device``, :meth:`from_synthetic`), which take no matrices themselves.
        A per-track ``R`` selects the generic update, as :meth:`from_tracks` with ``R`` does."""
        kw = {}
        for name, mats in (("Q", Q), ("R", R)):
            if mats is not None:
                pl = track_planes(name, mats, self.n_tracks)
                kw[name] = torch.from_numpy(np.ascontiguousarray(pl if self.order is None else pl[:, self.order])).to(self.device)
        return replace(self, **kw)

    # ------------------------------------------------------------------ #
    @classmethod
    def from_synthetic(cls, syn, substeps: int = 1, need_rows: Sequence[bool] = (True, True, False, False)):
        """Tile from :func:`synthetic.make_tracks` output living on the target device.  The step grid
        is ``generate_dts(dts, substeps)`` per track and the update cadence is every ``substeps``-th
        step, which is what the exact-equality rule yields for ``dts / k`` re-summed ``k`` times when
        ``k`` is a power of two (and for k = 1)."""
        if substeps < 1:
            raise ValueError("substeps must be >= 1")
        k = int(substeps)
        dts = syn.dts
        nobs = syn.nobs
        valid_gap = torch.arange(dts.shape[0], device=dts.device)[:, None] < (nobs.to(torch.int64) - 1)[None, :]
        if not bool(((dts > 0) | ~valid_gap).all().item()):
            raise ValueError("from_synthetic needs strictly positive gaps between fixes (the reference's update rule matches "
                             "accumulated times against np.cumsum(dts); use from_tracks for such data)")
        dt = (dts / k).repeat_interleave(k, dim=0).contiguous() if k > 1 else dts.contiguous()
        # "every k-th step" is what the reference's exact-equality rule gives when dts / k re-summed k
        # times is exact: k a power of two and the gaps on a 2^-10 h grid.  Anything else (k = 3, 6,
        # 7 ... or arbitrary gaps) gets its mask from the reference's own arithmetic, track by track.
        upd_mask = None
        exact = (k & (k - 1)) == 0 and bool((torch.round(dts * 1024.0) == dts * 1024.0).all().item())
        if not exact:
            dts_h, dt_h, nobs_h = dts.cpu().numpy(), dt.cpu().numpy(), nobs.cpu().numpy()
            mask = np.zeros(dt_h.shape, dtype=np.uint8)
            for t in range(dt_h.shape[1]):
                m = int(nobs_h[t])
                mk = exact_update_mask(dt_h[: (m - 1) * k, t], dts_h[: m - 1, t])
                if 1 + int(mk.sum()) > m:
                    raise IndexError(f"track {t}: {1 + int(mk.sum())} update times matched but only {m} observations")
                mask[: (m - 1) * k, t] = mk
            upd_mask = torch.from_numpy(mask).to(dts.device)
        uniform = bool((nobs == nobs[0]).all().item())
        n_steps = None if uniform else ((nobs - 1) * k).to(torch.int32).contiguous()
        rows = [syn.lon, syn.lat, syn.sog, syn.cog]
        z = [rows[r].contiguous() if need_rows[r] else None for r in range(4)]
        rate_rep, rate_rep_all = None, k
        nsteps_host = ((nobs - 1) * k).cpu().numpy()
        rep_host = ((nsteps_host + 1) // np.maximum(nobs.cpu().numpy() - 1, 1)).astype(np.int32)
        if np.all(rep_host == rep_host[0]):
            rate_rep_all = int(rep_host[0])
        else:
            rate_rep = torch.from_numpy(rep_host).to(syn.lon.device)
        return cls(
            x0=syn.x0().contiguous(), dt=dt, sog_rate=syn.sog_rate.contiguous(), cog_rate=syn.cog_rate.contiguous(),
            z=z, upd_mask=upd_mask, n_steps=n_steps, rate_repeat=rate_rep, substeps=k, rate_repeat_all=rate_rep_all,
            n_steps_host=nsteps_host,
        )

    @classmethod
    def from_tracks(
        cls,
        tracks: Sequence,
        dt_arrays: Sequence[np.ndarray],
        device="cuda",
        x0: Optional[Sequence[np.ndarray]] = None,
        time0: float = 0.0,
        noise: Optional[Sequence[Optional[Dict[str, np.ndarray]]]] = None,
        smoother: bool = True,
        sort_by_length: bool = True,
        R: Optional[Sequence[np.ndarray]] = None,
        Q: Optional[Sequence[np.ndarray]] = None,
    ):
        """Pack ``ShipTrack``-like objects (attributes ``dts, z, sog_rate, cog_rate``) with their step
        grids ``dt_arrays`` (what ``run(nsteps, dt, ship_track)`` receives).

        Ragged fleets are packed in order of decreasing length (``sort_by_length``; stable, so equal
        lengths keep the caller's order): the threads of a warp then finish together and a tile runs
        as long as its work, not as its longest track times its width.  ``TrackBatch.order`` records
        the permutation and ``TrackResults.track(i)`` undoes it - ``i`` is always the caller's index,
        and every track's numbers are bit-identical to the unsorted packing.  ``R``: one symmetric
        4 x 4 measurement covariance per track (instead of the filter's shared one).  ``Q``: one symmetric 4 x 4
        process noise matrix per track, in the caller's order, used by both passes instead of the filter's shared one:
        each track equals a filter built with its own ``Q``.  ``ValueError`` for a wrong count of either.

        Raises ``IndexError`` where the reference would: more matched observation times than
        observations (``kalman_filter.py:101-108``) or a smoother rate index past the repeated rate
        arrays (``unscented.py:287-311``).
        """
        T = len(tracks)
        if T == 0:
            raise ValueError("empty batch")
        Qt = None if Q is None else track_planes("Q", Q, T)
        dt_arrays = [np.asarray(d, dtype=np.float64).reshape(-1) for d in dt_arrays]
        order = length_order([len(d) for d in dt_arrays]) if sort_by_length else None
        if order is not None:
            tracks = [tracks[j] for j in order]
            dt_arrays = [dt_arrays[j] for j in order]
            x0 = None if x0 is None else [x0[j] for j in order]
            noise = None if noise is None else [noise[j] for j in order]
            R = None if R is None else [R[j] for j in order]
        nsteps = np.array([len(d) for d in dt_arrays], dtype=np.int32)
        nobs = np.array([np.asarray(tr.z).shape[1] for tr in tracks], dtype=np.int32)
        N, M = int(nsteps.max()), int(nobs.max())
        dt = np.zeros((max(N, 1), T))
        mask = np.zeros((max(N, 1), T), dtype=np.uint8)
        z = np.zeros((4, M, T))
        sr = np.zeros((M, T))
        cr = np.zeros((M, T))
        x0a = np.zeros((4, T))
        rep = np.ones(T, dtype=np.int32)
        for i, tr in enumerate(tracks):
            zi = np.asarray(tr.z, dtype=np.float64)
            if zi.shape[0] != 4:
                raise NotImplementedError("the CUDA path needs the 4-row measurement z = [lon; lat; sog; cog]")
            n, m = int(nsteps[i]), int(nobs[i])
            dt[:n, i] = dt_arrays[i]
            mask[:n, i] = track_update_mask(i, tr, dt_arrays[i], m, time0)
            z[:, :m, i] = zi
            sr[:m, i], cr[:m, i] = track_rates(i, tr, m)
            x0a[:, i] = zi[:, 0] if x0 is None else np.asarray(x0[i], dtype=np.float64).reshape(-1)
            if smoother:
                rep[i] = track_rate_repeat(i, tr, n, m)
        dev = torch.device(device)

        def up(a):
            return torch.from_numpy(np.ascontiguousarray(a)).to(dev)

        kw = {}
        if R is not None:
            Rt = np.stack([_as44("R", Ri) for Ri in R], axis=-1).reshape(16, T)
            if not np.array_equal(Rt.reshape(4, 4, T), Rt.reshape(4, 4, T).transpose(1, 0, 2)):
                raise NotImplementedError("per-track R must be symmetric for the CUDA path")
            kw["R"] = up(Rt)
        if Qt is not None:
            kw["Q"] = up(Qt if order is None else Qt[:, order])
        if noise is not None:
            npred = np.zeros((max(N, 1), 4, T))
            nupd = np.zeros((M, 4, T))
            nbwd = np.zeros((max(N, 1), 4, T))
            for i, nz in enumerate(noise):
                if nz is None:
                    continue
                if "pred" in nz and nz["pred"] is not None:
                    npred[: nsteps[i], :, i] = nz["pred"]
                if "upd" in nz and nz["upd"] is not None:
                    nupd[: len(nz["upd"]), :, i] = nz["upd"]
                if "bwd" in nz and nz["bwd"] is not None:
                    nbwd[: nsteps[i], :, i] = nz["bwd"]
            kw.update(noise_pred=up(npred), noise_upd=up(nupd), noise_bwd=up(nbwd))
        return cls(
            x0=up(x0a), dt=up(dt), sog_rate=up(sr), cog_rate=up(cr), z=[up(z[r]) for r in range(4)],
            upd_mask=up(mask), n_steps=up(nsteps), rate_repeat=up(rep), substeps=1, rate_repeat_all=1,
            n_steps_host=nsteps.copy(), order=order, **kw,
        )


@dataclass
class TrackResults:
    """Per-step states of a tile, in the kernels' layout: ``mean [N+1][4][T]``, ``cov [N+1][16][T]``."""

    mean_f: torch.Tensor
    cov_f: torch.Tensor
    mean_s: Optional[torch.Tensor]
    cov_s: Optional[torch.Tensor]
    status: torch.Tensor
    n_updates: torch.Tensor
    gate_iters: Optional[torch.Tensor] = None
    gate_lambda: Optional[torch.Tensor] = None
    gate_scale: Optional[torch.Tensor] = None
    smooth_stats: Optional[torch.Tensor] = None  # [N][15][T] device-side tape between the two passes (not a result)
    n_steps_host: Optional[np.ndarray] = None
    order: Optional[np.ndarray] = None  # TrackBatch.order of the tile these results belong to
    filtered_by: Optional[int] = field(default=None, repr=False, compare=False)  # id() of the tile last filtered into these buffers
    _column_of: Optional[np.ndarray] = field(default=None, repr=False, compare=False)
    # innovation statistics per update (allocate(..., innovations=True)), [max_obs][T], row = update index: y^T S^+ y, the
    # Gaussian log-likelihood of the update's observation and the rank of S^+ (include/ste_ukf.h, SteInnovations)
    nis: Optional[torch.Tensor] = None
    loglik: Optional[torch.Tensor] = None
    innov_rank: Optional[torch.Tensor] = None

    @property
    def packed_cov(self) -> bool:
        """True when the covariance tensors hold the 10 unique entries per state (``[N+1][10][T]``,
        order 00 01 02 03 11 12 13 22 23 33) instead of the full row-major 4x4."""
        return self.cov_f.shape[1] == 10

    @staticmethod
    def expand_cov(c: np.ndarray) -> np.ndarray:
        """``(..., 10)`` packed symmetric entries -> ``(..., 4, 4)``."""
        idx = np.array([[0, 1, 2, 3], [1, 4, 5, 6], [2, 5, 7, 8], [3, 6, 8, 9]])
        return c[..., idx]

    _TENSORS = ("mean_f", "cov_f", "mean_s", "cov_s", "status", "n_updates", "gate_iters", "gate_lambda", "gate_scale", "nis", "loglik",
                "innov_rank")

    def host_like(self, pinned: bool = True) -> "TrackResults":
        """Empty host buffers of the same shapes (page-locked by default) for device->host copies."""
        def mk(t):
            if t is None:
                return None
            h = torch.empty(t.shape, dtype=t.dtype, device="cpu")
            return h.pin_memory() if pinned else h
        kw = {n: mk(getattr(self, n)) for n in self._TENSORS}
        if self.mean_s is self.mean_f:
            kw["mean_s"], kw["cov_s"] = kw["mean_f"], kw["cov_f"]
        return TrackResults(n_steps_host=self.n_steps_host, order=self.order, **kw)

    def copy_to(self, other: "TrackResults", non_blocking: bool = True) -> int:
        """Copy every buffer into ``other`` (e.g. device -> pinned host); returns the bytes moved."""
        moved, seen = 0, set()
        for n in self._TENSORS:
            src, dst = getattr(self, n), getattr(other, n)
            if src is None or dst is None or dst.data_ptr() in seen:
                continue
            dst.copy_(src, non_blocking=non_blocking)
            seen.add(dst.data_ptr())
            moved += src.numel() * src.element_size()
        return moved

    def to_host(self, pinned: bool = False) -> "TrackResults":
        """Host copy of every buffer (one device->host transfer per array); ``track(i)`` on the copy
        costs no further transfers - the form the fleet writers use."""
        if not self.mean_f.is_cuda:
            return self
        host = self.host_like(pinned=pinned)
        self.copy_to(host, non_blocking=pinned)
        if pinned:
            torch.cuda.current_stream(self.mean_f.device).synchronize()
        return host

    def check_status(self, raise_on: int = nat.STE_STATUS_NONFINITE | nat.STE_STATUS_OBS_OVERRUN) -> Dict[str, int]:
        """Per-track status bits (``STE_STATUS_*``) summarised as counts; raises ``FloatingPointError``
        for non-finite states and ``IndexError`` for an observation overrun (where the reference
        raises, ``kalman_filter.py:101-108``) unless masked out of ``raise_on``."""
        st = self.status.cpu().numpy()
        names = {"nonfinite": nat.STE_STATUS_NONFINITE, "indefinite": nat.STE_STATUS_INDEFINITE, "gate_cap": nat.STE_STATUS_GATE_CAP,
                 "obs_overrun": nat.STE_STATUS_OBS_OVERRUN, "rank_deficient": nat.STE_STATUS_RANK_DEFICIENT,
                 "smooth_recompute": nat.STE_STATUS_SMOOTH_RECOMPUTE}
        counts = {k: int(np.count_nonzero(st & bit)) for k, bit in names.items()}
        if raise_on & nat.STE_STATUS_OBS_OVERRUN and counts["obs_overrun"]:
            col = int(np.flatnonzero(st & nat.STE_STATUS_OBS_OVERRUN)[0])
            raise IndexError(f"{counts['obs_overrun']} track(s) matched more update times than they have observations "
                             f"(first: column {col})")
        if raise_on & nat.STE_STATUS_NONFINITE and counts["nonfinite"]:
            col = int(np.flatnonzero(st & nat.STE_STATUS_NONFINITE)[0])
            raise FloatingPointError(f"{counts['nonfinite']} track(s) produced non-finite states (first: column {col})")
        return counts

    def _cov_np(self, cov: torch.Tensor, n: int, i: int) -> np.ndarray:
        c = cov[: n + 1, :, i].cpu().numpy()
        return self.expand_cov(c) if cov.shape[1] == 10 else c.reshape(n + 1, 4, 4)

    def column(self, i: int) -> int:
        """Column of the caller's track ``i`` (tiles are packed by decreasing length, ``order``)."""
        if self.order is None:
            return int(i)
        if self._column_of is None:
            self._column_of = np.empty(len(self.order), dtype=np.int64)
            self._column_of[self.order] = np.arange(len(self.order))
        return int(self._column_of[i])

    def track(self, i: int) -> Dict[str, np.ndarray]:
        """Host copies for the caller's track ``i`` in the reference's shapes: means (N+1, 4), covs (N+1, 4, 4)."""
        i = self.column(i)
        n = int(self.n_steps_host[i]) if self.n_steps_host is not None else self.mean_f.shape[0] - 1
        out = {
            "means": self.mean_f[: n + 1, :, i].cpu().numpy(),
            "covs": self._cov_np(self.cov_f, n, i),
            "status": int(self.status[i].item()),
            "n_updates": int(self.n_updates[i].item()),
        }
        if self.mean_s is not None:
            out["means_s"] = self.mean_s[: n + 1, :, i].cpu().numpy()
            out["covs_s"] = self._cov_np(self.cov_s, n, i)
        if self.gate_iters is not None:
            m = out["n_updates"]
            out["gate_iters"] = self.gate_iters[:m, i].cpu().numpy().astype(np.int32)
            out["gate_lambda"] = self.gate_lambda[:m, i].cpu().numpy()
            out["gate_scale"] = self.gate_scale[:m, i].cpu().numpy()
        if self.nis is not None:
            innovation_columns(self, out, i)
        return out


class BatchedUKF:
    """UKF forward filter + URTSS backward smoother over a :class:`TrackBatch` on one GPU.

    Results parity contract: every track equals a fresh reference ``UnscentedKalmanFilter`` run
    (``run`` then ``run_rts_smoother``) on the same inputs, with the reference's noise draws either
    zero or replayed from the batch's noise tapes.
    """

    def __init__(self, H, Q=None, R=None, P=None, *, gating=False, gate_chi=50.0, gate_max_iter=100, force_generic=False,
                 packed_cov=False, long_steps=None, measurement_model=None):
        if H is None:
            raise ValueError("Set proper system dynamics.")  # reference unscented.py:52-53
        eye = np.eye(4)
        self.model = FilterModel(
            H=H, Q=eye if Q is None else Q, R=eye if R is None else R, P0=eye if P is None else P,
            gating=gating, gate_chi=gate_chi, gate_max_iter=gate_max_iter, force_generic=force_generic,
        )
        self._lib = nat.load()
        # named element-wise transform of the observations before every update (reference unscented.py:221-225)
        from .measurement_models import MEASUREMENT_MODELS
        if measurement_model is not None and measurement_model not in MEASUREMENT_MODELS.values():
            raise NotImplementedError("measurement_model must be one of ship_track_estimators_b200.measurement_models."
                                      f"{sorted(MEASUREMENT_MODELS)} (arbitrary callables cannot run inside the kernels)")
        self.measurement_model = measurement_model
        # store the 10 unique covariance entries per state instead of the full 4x4 (30 % less state
        # traffic, memory and PCIe volume; TrackResults.track() expands them back)
        self.packed_cov = bool(packed_cov)
        # The geodetic step has a cheaper tier for displacements <= 100 km per predict, chosen per
        # step and track.  A tile that MIXES such steps with longer ones (sparse historical fixes
        # beside dense ones) makes the lanes of a warp run both tiers; STE_FLAG_LONG_STEPS keeps every
        # step on the full-range tier instead.  Results agree to 1 ulp either way.  None (default):
        # decided per tile from TrackBatch.long_step_fraction() (one cached device reduction the first
        # time a tile is launched); True / False pin the choice (no reduction, no synchronisation).
        self.long_steps = None if long_steps is None else bool(long_steps)
        self._pipe = None   # streams of run_host_pipelined, created once

    # ------------------------------------------------------------------ #
    def _problem(self, b: TrackBatch) -> nat.SteProblem:
        m = self.model
        p = nat.SteProblem()
        p.n_tracks, p.max_steps, p.max_obs = b.n_tracks, b.max_steps, b.max_obs
        p.substeps, p.rate_repeat = int(b.substeps), int(b.rate_repeat_all)
        p.flags = ((nat.STE_FLAG_GATING if m.gating else 0) | (nat.STE_FLAG_FORCE_GENERIC if (m.force_generic or b.R is not None) else 0)
                   | (nat.STE_FLAG_PACKED_COV if self.packed_cov else 0) | (nat.STE_FLAG_LONG_STEPS if self._long_steps_for(b) else 0))
        p.gate_max_iter, p.gate_chi = int(m.gate_max_iter), float(m.gate_chi)
        p.ld = b.n_tracks
        for name, M in (("H", m.H), ("Q", m.Q), ("R", m.R), ("P0", m.P0)):
            getattr(p, name)[:] = M.reshape(-1).tolist()
        return p

    #: a tile whose share of > 90 km legs lies between these bounds mixes the two geodetic tiers
    #: inside most warps and is pinned to the full-range tier
    LONG_STEP_MIX = (0.02, 1.0)

    def _long_steps_for(self, b: TrackBatch) -> bool:
        if self.long_steps is not None:
            return self.long_steps
        lo, hi = self.LONG_STEP_MIX
        return lo < b.long_step_fraction() <= hi

    def _inputs(self, b: TrackBatch) -> nat.SteInputs:
        i = nat.SteInputs()
        i.x0, i.P0, i.dt = nat.ptr(b.x0), nat.ptr(b.P0), nat.ptr(b.dt)
        i.upd_mask, i.n_steps = nat.ptr(b.upd_mask), nat.ptr(b.n_steps)
        rows = b.z
        if self.measurement_model is not None:
            cached = getattr(b, "_z_model", None)
            if cached is None or cached[0] is not self.measurement_model:
                from .measurement_models import apply_rows
                cached = b._z_model = (self.measurement_model, apply_rows(self.measurement_model, b.z))
            rows = cached[1]
        i.R_tracks = nat.ptr(b.R)
        for r in range(4):
            i.z[r] = nat.ptr(rows[r])
        i.sog_rate, i.cog_rate, i.rate_repeat = nat.ptr(b.sog_rate), nat.ptr(b.cog_rate), nat.ptr(b.rate_repeat)
        i.noise_pred, i.noise_upd, i.noise_bwd = nat.ptr(b.noise_pred), nat.ptr(b.noise_upd), nat.ptr(b.noise_bwd)
        return i

    def allocate(self, b: TrackBatch, smoother: bool = True, in_place: bool = False, reuse_stats: bool = True,
                 innovations: bool = False) -> TrackResults:
        """Output buffers for a tile (caller-owned, reusable across tiles of the same shape).

        ``reuse_stats``: also allocate the 240 B/step tape on which the forward pass leaves the
        smoother's sigma-point statistics, so the backward pass does not recompute them (the
        reference does).  ``False`` trades that memory for ~2x the smoother's arithmetic.
        ``innovations``: also allocate the ``nis`` / ``loglik`` / ``innov_rank`` planes ``[max_obs][T]``
        that the forward pass then fills per update (17 B per update; see :func:`allocate_innovations`)."""
        dev, T, S = b.device, b.n_tracks, b.max_steps + 1
        f64 = dict(dtype=torch.float64, device=dev)
        C = 10 if self.packed_cov else 16
        mean_f = torch.empty(S, 4, T, **f64)
        cov_f = torch.empty(S, C, T, **f64)
        mean_s = cov_s = None
        if smoother:
            mean_s, cov_s = (mean_f, cov_f) if in_place else (torch.empty(S, 4, T, **f64), torch.empty(S, C, T, **f64))
        res = TrackResults(
            mean_f=mean_f, cov_f=cov_f, mean_s=mean_s, cov_s=cov_s,
            status=torch.zeros(T, dtype=torch.int32, device=dev), n_updates=torch.zeros(T, dtype=torch.int32, device=dev),
            n_steps_host=b.n_steps_host, order=b.order,
        )
        if smoother and reuse_stats:
            res.smooth_stats = torch.empty(max(b.max_steps, 1), nat.STATS_PLANES, T, **f64)
        if self.model.gating:
            res.gate_iters = torch.zeros(b.max_obs, T, dtype=torch.uint8, device=dev)
            res.gate_lambda = torch.ones(b.max_obs, T, **f64)
            res.gate_scale = torch.ones(b.max_obs, T, **f64)
        if innovations:
            allocate_innovations(res, b.max_obs, T, dev)
        return res

    def _outputs(self, r: TrackResults) -> nat.SteOutputs:
        o = nat.SteOutputs()
        o.mean_f, o.cov_f = nat.ptr(r.mean_f), nat.ptr(r.cov_f)
        o.mean_s, o.cov_s = nat.ptr(r.mean_s), nat.ptr(r.cov_s)
        o.status, o.n_updates = nat.ptr(r.status), nat.ptr(r.n_updates)
        o.gate_iters, o.gate_lambda = nat.ptr(r.gate_iters), nat.ptr(r.gate_lambda)
        o.gate_scale = nat.ptr(r.gate_scale)
        o.smooth_stats = nat.ptr(r.smooth_stats)
        return o

    def _check_rows(self, b: TrackBatch):
        need_rows = [True] * 4 if b.R is not None else self.model.rows_needed()
        for r, need in enumerate(need_rows):
            if need and b.z[r] is None:
                raise ValueError(f"observation row {r} is referenced by H/R but absent from the batch")

    def _check_layout(self, res: TrackResults):
        if res.packed_cov != self.packed_cov:
            raise ValueError("result buffers were allocated with a different covariance layout (packed_cov)")

    def _check_shapes(self, b: TrackBatch, res: TrackResults, smoother: bool = False) -> None:
        """The kernels receive raw pointers: every buffer of ``res`` must have been allocated for a
        tile of exactly ``b``'s shape (``allocate(b)``), on ``b``'s device."""
        b.check()
        self._check_layout(res)
        T, S, dev = b.n_tracks, b.max_steps + 1, b.device
        planes = 10 if self.packed_cov else 16
        expect = [("mean_f", res.mean_f, (S, 4, T)), ("cov_f", res.cov_f, (S, planes, T)), ("status", res.status, (T,)),
                  ("n_updates", res.n_updates, (T,))]
        if smoother:
            if res.mean_s is None or res.cov_s is None:
                raise ValueError("results were allocated without smoother buffers")
            expect += [("mean_s", res.mean_s, (S, 4, T)), ("cov_s", res.cov_s, (S, planes, T))]
        if res.smooth_stats is not None:
            expect.append(("smooth_stats", res.smooth_stats, (max(b.max_steps, 1), nat.STATS_PLANES, T)))
        for name in ("gate_iters", "gate_lambda", "gate_scale"):
            if getattr(res, name) is not None:
                expect.append((name, getattr(res, name), (b.max_obs, T)))
        for name, t, shape in expect:
            if t is None or tuple(t.shape) != shape or t.device != dev or not t.is_contiguous():
                got = "None" if t is None else f"{tuple(t.shape)} on {t.device}"
                raise ValueError(f"TrackResults.{name}: expected a contiguous tensor of shape {shape} on {dev} for this tile, got {got}")
        check_innovations(res, "TrackResults", b.max_obs, T, dev)
        if self.model.gating and res.gate_iters is None:
            raise ValueError("results were allocated without gating buffers (allocate() with a gating model)")

    def forward(self, b: TrackBatch, res: TrackResults) -> None:
        """Launch the forward filter (asynchronous on the current stream)."""
        self._check_rows(b)
        self._check_shapes(b, res)
        if self.model.gating and b.noise_upd is not None:
            raise NotImplementedError("gating with measurement noise tapes (data-dependent draw count)")
        p, i, o = self._problem(b), self._inputs(b), self._outputs(res)
        res.filtered_by = id(b)
        with torch.cuda.device(b.device):
            if b.Q is not None:
                innov = None if res.nis is None else C.byref(innovation_planes(res))
                nat.check(self._lib.ste_ukf_forward_noise_f64(C.byref(p), C.byref(i), C.byref(self._noise(b)), innov, C.byref(o),
                                                              nat.current_stream()))
            elif res.nis is None:
                nat.check(self._lib.ste_ukf_forward_f64(C.byref(p), C.byref(i), C.byref(o), nat.current_stream()))
            else:
                nat.check(self._lib.ste_ukf_forward_innov_f64(C.byref(p), C.byref(i), C.byref(innovation_planes(res)), C.byref(o),
                                                              nat.current_stream()))

    def backward(self, b: TrackBatch, res: TrackResults) -> None:
        """Launch the URTSS backward pass over the filtered states in ``res``."""
        self._check_shapes(b, res, smoother=True)
        self._check_filtered(b, res)
        p, i, o = self._problem(b), self._inputs(b), self._outputs(res)
        with torch.cuda.device(b.device):
            if b.Q is not None:
                nat.check(self._lib.ste_urtss_backward_noise_f64(C.byref(p), C.byref(i), C.byref(self._noise(b)), C.byref(o),
                                                                 nat.current_stream()))
            else:
                nat.check(self._lib.ste_urtss_backward_f64(C.byref(p), C.byref(i), C.byref(o), nat.current_stream()))

    @staticmethod
    def _noise(b: TrackBatch) -> nat.SteNoiseN:
        """The per-track process noise of ``b`` (the n = 4 passes take a per-track ``R`` in ``SteInputs.R_tracks``)."""
        return nat.SteNoiseN(nat.ptr(b.Q), None)

    @staticmethod
    def _check_filtered(b: TrackBatch, res: TrackResults) -> None:
        """The backward pass reads the filtered states, status bits and statistics tape the forward
        pass of THE SAME tile left in ``res``; a stale tape from another tile would be used silently."""
        by = getattr(res, "filtered_by", None)
        if by is not None and by != id(b):
            raise ValueError("these results were last filtered from a different tile: run forward() on this tile first")

    def fused(self, fwd_batch: TrackBatch, fwd_res: TrackResults, bwd_batch: TrackBatch, bwd_res: TrackResults) -> None:
        """ONE launch: the forward filter of ``fwd_batch`` and the backward smoother of ``bwd_batch``
        (filtered by an earlier ``forward``/``fused`` call into ``bwd_res``), as blocks of two roles
        resident on every SM together.  Bit-identical to ``forward(fwd_batch, fwd_res);
        backward(bwd_batch, bwd_res)``, and on B200 ~13 % slower than those two launches (two
        instruction streams per SM overflow the instruction cache).  The two result sets must be distinct.
        The fused launch writes no innovation statistics and takes no per-track ``Q``: ``fwd_res`` with innovation planes,
        or a tile with ``TrackBatch.Q``, raises ``ValueError``."""
        if fwd_res.nis is not None:
            raise ValueError("the fused pass writes no innovation statistics: filter tiles with innovation planes with forward()")
        if fwd_batch.Q is not None or bwd_batch.Q is not None:
            raise ValueError("the fused pass takes no per-track Q: run tiles with TrackBatch.Q with forward() / backward()")
        self._check_rows(fwd_batch)
        self._check_shapes(fwd_batch, fwd_res)
        self._check_shapes(bwd_batch, bwd_res, smoother=True)
        self._check_filtered(bwd_batch, bwd_res)
        if self.model.gating and fwd_batch.noise_upd is not None:
            raise NotImplementedError("gating with measurement noise tapes (data-dependent draw count)")
        if fwd_batch.device != bwd_batch.device:
            raise ValueError("both tiles of a fused pass must live on one device")
        pf, i_f, of = self._problem(fwd_batch), self._inputs(fwd_batch), self._outputs(fwd_res)
        pb, ib, ob = self._problem(bwd_batch), self._inputs(bwd_batch), self._outputs(bwd_res)
        fwd_res.filtered_by = id(fwd_batch)
        with torch.cuda.device(fwd_batch.device):
            nat.check(self._lib.ste_ukf_fused_f64(C.byref(pf), C.byref(i_f), C.byref(of), C.byref(pb), C.byref(ib), C.byref(ob),
                                                  nat.current_stream()))

    def run_many(self, batches: Sequence[TrackBatch], results: Sequence[TrackResults], fused: bool = False,
                 partition=None) -> None:
        """Filter and smooth a sequence of resident tiles.  Default: two launches per tile.
        ``partition=SmPartition(...)`` (``partition.py``): software-pipelined on disjoint SMs - tile i+1
        is filtered on the partition's filter stream while tile i is smoothed on its smoother stream
        (the same two kernels, bit-identical results; ~6 % more tiles per second on a B200).
        ``fused=True``: tile i+1 is filtered by the same launch that smooths tile i
        (``len(batches) + 1`` launches; measured slower than two launches, kept for reference).
        With either pipelined schedule consecutive tiles must use different result sets (two
        alternating sets are enough when each tile's results are consumed, in stream order, before
        its set comes round again)."""
        n = len(batches)
        if n != len(results):
            raise ValueError("one result set per tile")
        if partition is not None:
            if fused:
                raise ValueError("choose one of fused=True and partition=...")
            return self._run_many_partitioned(batches, results, partition)
        if fused and any(b.Q is not None for b in batches):
            raise ValueError("the fused pass takes no per-track Q: run tiles with TrackBatch.Q with forward() / backward()")
        if not fused:
            for b, r in zip(batches, results):
                self.forward(b, r)
                self.backward(b, r)
            return
        for i in range(n + 1):
            if i == 0:
                self.forward(batches[0], results[0])
            elif i == n:
                self.backward(batches[n - 1], results[n - 1])
            else:
                self.fused(batches[i], results[i], batches[i - 1], results[i - 1])

    def _run_many_partitioned(self, batches, results, part) -> None:
        """forward(tile i) on ``part.filter_stream`` beside backward(tile i-1) on ``part.smoother_stream``.
        Ordering by events: a tile is smoothed after its own filter pass, and a result set is written by
        the next filter pass only after the smoother pass that last used it.  Returns with the caller's
        current stream waiting on both."""
        n = len(batches)
        for i in range(1, n):
            if results[i] is results[i - 1]:
                raise ValueError("consecutive tiles need different result sets on the partitioned schedule")
        dev = results[0].mean_f.device if n else None
        if n == 0:
            return
        cur = torch.cuda.current_stream(dev)
        fs, bs = part.filter_stream, part.smoother_stream
        fs.wait_stream(cur)
        bs.wait_stream(cur)
        smoothed = {}   # id(result set) -> event after the smoother pass that last used it
        filtered = None
        for i in range(n + 1):
            ev_f = None
            if i < n:
                last = smoothed.pop(id(results[i]), None)
                if last is not None:
                    fs.wait_event(last)
                with torch.cuda.stream(fs):
                    self.forward(batches[i], results[i])
                    ev_f = torch.cuda.Event()
                    ev_f.record(fs)
            if i >= 1:
                bs.wait_event(filtered)
                with torch.cuda.stream(bs):
                    self.backward(batches[i - 1], results[i - 1])
                    ev_b = torch.cuda.Event()
                    ev_b.record(bs)
                smoothed[id(results[i - 1])] = ev_b
            filtered = ev_f
        cur.wait_stream(fs)
        cur.wait_stream(bs)

    # ------------------------------------------------------------------ #
    # host-buffer (end-to-end) entry points                              #
    # ------------------------------------------------------------------ #
    #: named selections of what travels back to the host per tile.  Per stored state: "all" 224 B
    #: (packed covariances; 320 B full), "cli" 128 B - what the reference CLI writes, means and
    #: diag(P) of the filtered and the smoothed pass (main_cli.py:146-167) -, "smoothed" 64 B - the
    #: smoothed track with its variances -, "summary" nothing per state: per track the last filtered
    #: state and the fit metrics of performance_metrics.track_metrics.
    OUTPUT_SETS = {
        "all": ("mean_f", "cov_f", "mean_s", "cov_s"),
        "cli": ("mean_f", "diag_f", "mean_s", "diag_s"),
        "filtered": ("mean_f", "diag_f"),
        "smoothed": ("mean_s", "diag_s"),
        "summary": ("final", "metrics"),
    }

    def _output_names(self, outputs, smoother: bool):
        return output_names(self.OUTPUT_SETS, outputs, smoother)

    def host_outputs(self, b: TrackBatch, outputs="all", smoother: bool = True, pinned: bool = True) -> Dict[str, torch.Tensor]:
        """Host buffers (page-locked by default) for the selected outputs of a tile shaped like ``b``,
        plus the always-returned per-track ``status`` and ``n_updates``."""
        T, S, C_ = b.n_tracks, b.max_steps + 1, (10 if self.packed_cov else 16)
        shapes = {"mean_f": (S, 4, T), "mean_s": (S, 4, T), "cov_f": (S, C_, T), "cov_s": (S, C_, T), "diag_f": (S, 4, T),
                  "diag_s": (S, 4, T), "final": (4 + C_, T), "metrics": (12, T)}
        out = {}
        for n in self._output_names(outputs, smoother) + ("status", "n_updates"):
            t = torch.empty(shapes.get(n, (T,)), dtype=torch.int32 if n in ("status", "n_updates") else torch.float64)
            out[n] = t.pin_memory() if pinned else t
        return out

    def _extract(self, b: TrackBatch, res: TrackResults, names, smoother: bool, scratch: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        """Device tensors for the selected outputs (views where the result buffers already hold them,
        small gathers into ``scratch`` otherwise)."""
        dev = b.device
        dsel = scratch.get("_diag_idx")
        if dsel is None:
            dsel = scratch["_diag_idx"] = torch.tensor([0, 4, 7, 9] if self.packed_cov else [0, 5, 10, 15], device=dev)
        out = {"status": res.status, "n_updates": res.n_updates}
        for n in names:
            if n in ("mean_f", "cov_f", "mean_s", "cov_s"):
                out[n] = getattr(res, n)
            elif n in ("diag_f", "diag_s"):
                cov = res.cov_f if n == "diag_f" else res.cov_s
                buf = scratch.get(n)
                if buf is None or buf.shape != (cov.shape[0], 4, cov.shape[2]):
                    buf = scratch[n] = torch.empty(cov.shape[0], 4, cov.shape[2], dtype=torch.float64, device=dev)
                torch.index_select(cov, 1, dsel, out=buf)
                out[n] = buf
            elif n == "final":
                if b.n_steps is None:
                    out[n] = torch.cat([res.mean_f[-1], res.cov_f[-1]], dim=0)
                else:
                    last = b.n_steps.to(torch.int64)[None, None, :]
                    out[n] = torch.cat([torch.gather(res.mean_f, 0, last.expand(1, 4, -1))[0],
                                        torch.gather(res.cov_f, 0, last.expand(1, res.cov_f.shape[1], -1))[0]], dim=0)
            elif n == "metrics":
                from .performance_metrics import track_metrics

                m = track_metrics(self, b, res, which="smoothed" if smoother else "filtered")
                out[n] = torch.cat([m["rmse"], m["cum_abs"], m["max_abs"]], dim=0)
        return out

    def run_host(self, host_batch: TrackBatch, host_out, dev_res: Optional[TrackResults] = None, smoother: bool = True,
                 device="cuda", outputs="all") -> Dict[str, int]:
        """End-to-end call on HOST buffers: pinned inputs -> device, forward (+ backward), the selected
        ``outputs`` -> pinned ``host_out`` (a dict from :meth:`host_outputs`, or a ``TrackResults`` of
        host tensors for ``outputs="all"``).  Asynchronous on the current stream; synchronise before
        reading ``host_out``.  Returns the bytes copied in each direction."""
        names = self._output_names(outputs, smoother)
        dev_batch = host_batch.to(device, non_blocking=True)
        dev_res = self.run(dev_batch, smoother=smoother, res=dev_res)
        d2h = copy_out(self._extract(dev_batch, dev_res, names, smoother, {}), host_out)
        return {"h2d_bytes": host_batch.input_bytes(), "d2h_bytes": d2h}

    def run_host_pipelined(self, host_batches: Sequence[TrackBatch], host_outs: Sequence, smoother: bool = True,
                           device="cuda", outputs="all") -> Dict[str, int]:
        """End-to-end over a sequence of HOST tiles with the three engines overlapped: while tile i
        is filtered and smoothed, tile i+1's inputs travel host->device and tile i-1's results
        device->host (PCIe is full duplex and the copy engines run beside the SMs).  Two device
        buffer sets alternate.  ``host_batches`` / ``host_outs`` live in pinned memory
        (``host_outs[i]``: a dict from :meth:`host_outputs`, or a host ``TrackResults`` for
        ``outputs="all"``); all tiles must share one shape.  ``outputs`` selects what is copied back
        (``OUTPUT_SETS``): PCIe carries ~50 GB/s, so the bytes per state decide the end-to-end rate.
        Returns the bytes copied over all tiles in each direction; synchronise before reading ``host_outs``."""
        return run_host_pipelined(self, host_batches, host_outs, self._output_names(outputs, smoother), smoother, device,
                                  layout=self.packed_cov)

    def score(self, b: TrackBatch, candidates: Sequence) -> Dict[str, torch.Tensor]:
        """Log-likelihood scores of noise candidates for every track of ``b``, without storing any state.

        ``candidates`` is a sequence of ``(Q, R)`` pairs, each checked as the constructor checks its own (4 x 4,
        symmetric) and finite.  Candidate ``c`` is scored as this filter with ``Q, R = candidates[c]`` would run
        ``run(b, smoother=False, innovations=True)``: its ``loglik`` / ``nis`` / ``dof`` / ``n_updates`` equal
        ``performance_metrics.innovation_metrics`` of that run, bit for bit, and ``status`` its status.  Returns those
        five device tensors ``[C][T]`` in the tile's column order (column j is the caller's track ``b.order[j]``).

        Candidates whose ``R`` selects the position-only update and those that need the generic one are launched
        apart; each launch covers up to ``STE_MAX_CANDIDATES`` candidates (asynchronous on the current stream).  A tile
        with its own per-track ``R`` or ``Q`` raises ``ValueError``: the candidates replace them."""
        b.check()
        if b.R is not None:
            raise ValueError("TrackBatch.R: a tile with per-track measurement noise cannot be scored (the candidates replace R)")
        if b.Q is not None:
            raise ValueError("TrackBatch.Q: a tile with per-track process noise cannot be scored (the candidates replace Q)")
        if self.model.gating and b.noise_upd is not None:
            raise NotImplementedError("gating with measurement noise tapes (data-dependent draw count)")
        m = self.model
        models = []
        for c, (Qc, Rc) in enumerate(candidate_pairs(candidates)):
            mc = FilterModel(H=m.H, Q=Qc, R=Rc, P0=m.P0, gating=m.gating, gate_chi=m.gate_chi, gate_max_iter=m.gate_max_iter,
                             force_generic=m.force_generic)
            if not (np.all(np.isfinite(mc.Q)) and np.all(np.isfinite(mc.R))):
                raise ValueError(f"candidate {c}: Q and R must be finite")
            for r, need in enumerate(mc.rows_needed()):
                if need and b.z[r] is None:
                    raise ValueError(f"candidate {c}: observation row {r} is referenced by H/R but absent from the batch")
            models.append(mc)
        pos = [mc.position_only() for mc in models]
        groups = [[c for c in range(len(models)) if pos[c] == v] for v in (True, False)]
        Q = np.stack([mc.Q.reshape(-1) for mc in models])
        R = np.stack([mc.R.reshape(-1) for mc in models])
        p, i = self._problem(b), self._inputs(b)
        with torch.cuda.device(b.device):
            return launch_scores(self._lib.ste_ukf_score_f64, p, i, [g for g in groups if g], Q, R, b.device)

    def run(self, b: TrackBatch, smoother: bool = True, res: Optional[TrackResults] = None, in_place: bool = False,
            innovations: bool = False) -> TrackResults:
        """Filter (and smooth) a tile into ``res`` or new buffers; ``innovations=True`` allocates the innovation
        statistics planes with them (``allocate``)."""
        res = res if res is not None else self.allocate(b, smoother=smoother, in_place=in_place, innovations=innovations)
        self.forward(b, res)
        if smoother:
            self.backward(b, res)
        return res


# ---------------------------------------------------------------------- #
# innovation statistics planes, shared by TrackResults and TrackResultsN  #
# ---------------------------------------------------------------------- #
def allocate_innovations(res, max_obs: int, T: int, dev) -> None:
    """Give ``res`` the ``nis`` / ``loglik`` (float64, NaN until written) and ``innov_rank`` (uint8) planes ``[max_obs][T]``."""
    res.nis = torch.full((max_obs, T), float("nan"), dtype=torch.float64, device=dev)
    res.loglik = torch.full((max_obs, T), float("nan"), dtype=torch.float64, device=dev)
    res.innov_rank = torch.zeros(max_obs, T, dtype=torch.uint8, device=dev)


def check_innovations(res, what: str, max_obs: int, T: int, dev) -> None:
    """All three innovation planes or none, each a contiguous ``[max_obs][T]`` tensor of its dtype on ``dev``."""
    planes = (("nis", torch.float64), ("loglik", torch.float64), ("innov_rank", torch.uint8))
    present = [getattr(res, n) is not None for n, _ in planes]
    if any(present) and not all(present):
        raise ValueError(f"{what}: nis, loglik and innov_rank are allocated together (allocate(..., innovations=True))")
    if not any(present):
        return
    for name, dtype in planes:
        t = getattr(res, name)
        if tuple(t.shape) != (max_obs, T) or t.dtype != dtype or t.device != dev or not t.is_contiguous():
            raise ValueError(f"{what}.{name}: expected a contiguous {dtype} tensor of shape {(max_obs, T)} on {dev} for this tile, "
                             f"got {t.dtype} {tuple(t.shape)} on {t.device}")


def innovation_planes(res) -> nat.SteInnovations:
    return nat.SteInnovations(nat.ptr(res.nis), nat.ptr(res.loglik), nat.ptr(res.innov_rank))


def innovation_columns(res, out: Dict[str, np.ndarray], j: int) -> None:
    """The innovation statistics of column ``j``'s ``out["n_updates"]`` updates into ``out``."""
    m = out["n_updates"]
    out["nis"] = res.nis[:m, j].cpu().numpy()
    out["loglik"] = res.loglik[:m, j].cpu().numpy()
    out["innov_rank"] = res.innov_rank[:m, j].cpu().numpy().astype(np.int32)


# ---------------------------------------------------------------------- #
# noise-candidate scores, shared by BatchedUKF.score and BatchedUKFN.score #
# ---------------------------------------------------------------------- #
SCORE_KEYS = ("loglik", "nis", "dof", "n_updates", "status")


def candidate_pairs(candidates: Sequence) -> List[tuple]:
    """``candidates`` as a list of ``(Q, R)`` pairs; ``ValueError`` for an empty sequence or an entry that is not a pair."""
    pairs = list(candidates)
    if not pairs:
        raise ValueError("no noise candidates to score")
    for c, pair in enumerate(pairs):
        if len(pair) != 2:
            raise ValueError(f"candidate {c}: expected a (Q, R) pair")
    return pairs


def launch_scores(fn, p, i, groups: Sequence[Sequence[int]], Q: np.ndarray, R: np.ndarray, dev) -> Dict[str, torch.Tensor]:
    """Score candidates ``Q[c]`` / ``R[c]`` (rows of row-major n x n entries) with the C entry point ``fn``
    (``ste_ukf_score_f64`` / ``ste_ukf_score_n_f64``) on problem ``p`` and inputs ``i``: one launch per chunk of at
    most ``STE_MAX_CANDIDATES`` candidates of each group (a list of candidate indices).  Returns the ``SCORE_KEYS`` tensors ``[C][T]``."""
    n_cand, T = len(Q), int(p.n_tracks)
    f64, i32 = dict(dtype=torch.float64, device=dev), dict(dtype=torch.int32, device=dev)
    out = {"loglik": torch.empty(n_cand, T, **f64), "nis": torch.empty(n_cand, T, **f64), "dof": torch.empty(n_cand, T, **i32),
           "n_updates": torch.empty(n_cand, T, **i32), "status": torch.empty(n_cand, T, **i32)}
    if T == 0:
        return out
    for group in groups:
        for lo in range(0, len(group), nat.STE_MAX_CANDIDATES):
            sel = list(group[lo: lo + nat.STE_MAX_CANDIDATES])
            rows = slice(sel[0], sel[0] + len(sel))
            direct = sel == list(range(rows.start, rows.stop))   # consecutive candidates are written in place
            dst = {k: v[rows] if direct else torch.empty(len(sel), T, dtype=v.dtype, device=dev) for k, v in out.items()}
            Qh, Rh = np.ascontiguousarray(Q[sel], dtype=np.float64), np.ascontiguousarray(R[sel], dtype=np.float64)
            dp = C.POINTER(C.c_double)
            cand = nat.SteCandidates(len(sel), 0, Qh.ctypes.data_as(dp), Rh.ctypes.data_as(dp))
            sc = nat.SteScores(*(nat.ptr(dst[k]) for k in SCORE_KEYS), T)
            nat.check(fn(C.byref(p), C.byref(i), C.byref(cand), C.byref(sc), nat.current_stream()))
            if not direct:
                idx = torch.tensor(sel, dtype=torch.int64, device=dev)
                for k, v in out.items():
                    v.index_copy_(0, idx, dst[k])
    return out


# ---------------------------------------------------------------------- #
# host-buffer entry points shared by BatchedUKF and batch_n.BatchedUKFN   #
# ---------------------------------------------------------------------- #
def output_names(output_sets: Dict[str, tuple], outputs, smoother: bool) -> tuple:
    """The output names of a set name of ``output_sets`` or an explicit list; unknown names and smoothed outputs
    without the smoother raise ``ValueError``."""
    names = output_sets[outputs] if isinstance(outputs, str) else tuple(outputs)
    known = {"mean_f", "cov_f", "mean_s", "cov_s", "diag_f", "diag_s", "final", "metrics"}
    for n in names:
        if n not in known:
            raise ValueError(f"unknown output {n!r}; choose from {sorted(known)} or a set name {sorted(output_sets)}")
        if not smoother and n.endswith("_s"):
            raise ValueError(f"output {n!r} needs the smoother")
    return names


def copy_out(dev_out: Dict[str, torch.Tensor], host_out) -> int:
    """Asynchronous device->host copies of ``dev_out`` into the same names of ``host_out`` (a dict or a host results
    object); returns the bytes moved."""
    moved = 0
    for n, src in dev_out.items():
        dst = host_out.get(n) if isinstance(host_out, dict) else getattr(host_out, n, None)
        if dst is None:
            continue
        dst.copy_(src, non_blocking=True)
        moved += src.numel() * src.element_size()
    return moved


def run_host_pipelined(engine, host_batches: Sequence, host_outs: Sequence, names: tuple, smoother: bool, device,
                       layout=None) -> Dict[str, int]:
    """The three-stream loop of ``run_host_pipelined`` for an engine with ``allocate`` / ``run`` / ``_extract`` and a
    ``_pipe`` slot, over tiles with ``copy_from`` / ``to`` / ``input_bytes``.  ``layout``: whatever else decides the
    shape of the engine's result buffers (kept with the tile shape to reuse them across calls)."""
    dev = torch.device(device)
    n = len(host_batches)
    if n != len(host_outs):
        raise ValueError("one host output set per tile")
    shape0 = (host_batches[0].n_tracks, host_batches[0].max_steps, host_batches[0].max_obs) if n else None
    for hb in host_batches:
        if (hb.n_tracks, hb.max_steps, hb.max_obs) != shape0:
            raise ValueError("run_host_pipelined: all tiles must share one shape (n_tracks, max_steps, max_obs); "
                             f"got {(hb.n_tracks, hb.max_steps, hb.max_obs)} after {shape0}")
    cur = torch.cuda.current_stream(dev)
    if engine._pipe is None or engine._pipe["device"] != dev:
        engine._pipe = {"device": dev, "streams": [torch.cuda.Stream(dev) for _ in range(3)], "res": [None, None],
                        "in": [None, None], "scratch": [{}, {}], "shape": None}
    pipe = engine._pipe
    key = (shape0, smoother, layout)
    if pipe["shape"] != key:                 # device input and result buffers are kept across calls of one shape
        pipe["res"], pipe["in"], pipe["scratch"], pipe["shape"] = [None, None], [None, None], [{}, {}], key
    s_in, s_run, s_out = pipe["streams"]
    for s_ in (s_in, s_run, s_out):
        s_.wait_stream(cur)
    dev_in: List = pipe["in"]    # two resident input tiles, overwritten in place (no allocation in the loop)
    in_done = [torch.cuda.Event() for _ in range(n)]
    run_done = [torch.cuda.Event() for _ in range(n)]
    out_done = [torch.cuda.Event() for _ in range(n)]
    moved = {"h2d_bytes": 0, "d2h_bytes": 0}
    for i in range(n):
        k = i % 2
        with torch.cuda.stream(s_in):
            if i >= 2:
                s_in.wait_event(run_done[i - 2])        # the kernels that read this input slot are done
            if dev_in[k] is None or not dev_in[k].copy_from(host_batches[i]):
                dev_in[k] = host_batches[i].to(dev, non_blocking=True)
            in_done[i].record(s_in)
        with torch.cuda.stream(s_run):
            s_run.wait_event(in_done[i])
            if i >= 2:
                s_run.wait_event(out_done[i - 2])       # this result slot has been copied out
            if pipe["res"][k] is None:
                pipe["res"][k] = engine.allocate(dev_in[k], smoother=smoother)
            res = pipe["res"][k]
            res.n_steps_host, res.order = dev_in[k].n_steps_host, dev_in[k].order
            engine.run(dev_in[k], smoother=smoother, res=res)
            dev_out = engine._extract(dev_in[k], res, names, smoother, pipe["scratch"][k])
            run_done[i].record(s_run)
        with torch.cuda.stream(s_out):
            s_out.wait_event(run_done[i])
            moved["d2h_bytes"] += copy_out(dev_out, host_outs[i])
            out_done[i].record(s_out)
        moved["h2d_bytes"] += host_batches[i].input_bytes()
    for s_ in (s_in, s_run, s_out):
        cur.wait_stream(s_)
    return moved
