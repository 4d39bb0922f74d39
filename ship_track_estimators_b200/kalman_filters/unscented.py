"""Unscented Kalman Filter with the reference's class API, executed on the GPU.

Drop-in for reference ``src/track_estimators/kalman_filters/unscented.py`` (Cole & Schamberg,
Applied Ocean Research 124 (2022) 103205).  Every arithmetic entry point - ``predict``, ``update``,
``run``, ``rts_step`` / ``run_rts_smoother``, ``compute_sigma_points``, ``check_robustness`` - is a
call into ``libste_ukf.so`` on a batch of one track; the many-track entry point is
:class:`ship_track_estimators_b200.batch.BatchedUKF`.  There is no host implementation: without
the CUDA library or a GPU these methods raise.

Noise.  The reference perturbs the predicted mean, the measurement and the back-predicted mean
with fresh ``np.random.normal`` draws (``unscented.py:198-202, 232-236, 320-323``).  This class
draws the same number of *unit* normals from the same global numpy generator in the same order and
lets the kernels scale them by ``sqrt(diag Q)`` / ``sqrt(diag R)``, so a seeded or monkey-patched
``np.random.normal`` pins both implementations identically.  ``noise="zero"`` (constructor or
``UnscentedKalmanFilter.default_noise``) disables the draws.
"""
from __future__ import annotations

import ctypes as C
import logging
from typing import Callable, Optional

import numpy as np

from .kalman_filter import KalmanFilterBase
from .non_linear_process import DEVICE_MODELS, geodetic_dynamics


def _unit_normals(rows: int, n: int) -> np.ndarray:
    """``rows`` successive ``np.random.normal(size=n)`` draws (same stream order as the reference)."""
    if rows == 0:
        return np.zeros((0, n))
    return np.asarray(np.random.normal(size=(rows, n)), dtype=np.float64).reshape(rows, n)


class _Stage:
    """Staging of a single-step call: ONE pinned host buffer, ONE device buffer, so that a `predict` or
    `update` costs one host->device copy, one launch and one device->host copy (the first round-2
    version made ~8 small allocations and 5 synchronous copies per call).  ``slot(name)`` hands out
    consecutive float64 ranges; the last one doubles as the int32 status word."""

    def __init__(self, layout):
        import torch

        self.offsets, n = {}, 0
        for name, size in layout:
            self.offsets[name] = (n, n + size)
            n += size
        self.host = torch.zeros(n, dtype=torch.float64).pin_memory()
        self.dev = torch.zeros(n, dtype=torch.float64, device="cuda")
        self.np = self.host.numpy()

    def put(self, name, values):
        a, b = self.offsets[name]
        self.np[a:b] = np.asarray(values, dtype=np.float64).reshape(-1)

    def get(self, name):
        a, b = self.offsets[name]
        return self.np[a:b].copy()

    def dev_slot(self, name):
        a, b = self.offsets[name]
        return self.dev[a:b]

    def upload(self, upto):
        self.dev[: self.offsets[upto][1]].copy_(self.host[: self.offsets[upto][1]], non_blocking=True)

    def download(self):
        import torch

        self.host.copy_(self.dev, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def status(self):
        a, _ = self.offsets["status"]
        return int(self.host[a:a + 1].view(torch_int32())[0])


def torch_int32():
    import torch

    return torch.int32


class UnscentedKalmanFilter(KalmanFilterBase):
    default_noise = "numpy"  # "numpy": reference semantics; "zero": deterministic

    def __init__(
        self,
        H=None,
        Q=None,
        R=None,
        P=None,
        x0=None,
        non_linear_process: Optional[Callable] = None,
        measurement_model: Optional[Callable] = None,
        *,
        gating: bool = False,
        noise: Optional[str] = None,
    ):
        """Same parameters as the reference (``unscented.py:20-74``); ``gating`` re-enables the
        Mahalanobis robustification the reference leaves commented out (``:228``)."""
        super().__init__()
        if H is None:
            raise ValueError("Set proper system dynamics.")
        self.H = H
        self.n = H.shape[1]
        self.Q = np.eye(self.n) if Q is None else np.asarray(Q)
        self.R = np.eye(self.n) if R is None else np.asarray(R)
        self.P_orig = np.eye(self.n) if P is None else np.asarray(P)
        self.P = np.eye(self.n) if P is None else np.asarray(P)
        self.x = np.zeros((self.n, 1)) if x0 is None else np.asarray(x0).reshape(-1, 1)

        self.n_sigma_points = 2 * self.n + 1
        self.sigma_points = np.zeros((self.n, self.n_sigma_points))
        self.sigma_points_orig = None
        self.weights = np.zeros((self.n_sigma_points, self.n_sigma_points))

        self.non_linear_process = non_linear_process
        self.measurement_model = measurement_model
        self.gating = bool(gating)
        self.noise = noise
        self.status = 0  # OR of STE_STATUS_* bits seen by this filter
        self._stages: dict = {}  # pinned / device staging buffers of the single-step calls, allocated once
        self.gate_iters: list = []
        self.gate_lambda: list = []

    # ------------------------------------------------------------------ #
    # helpers                                                            #
    # ------------------------------------------------------------------ #
    def _noise_on(self) -> bool:
        mode = self.noise if self.noise is not None else type(self).default_noise
        if mode not in ("numpy", "zero"):
            raise ValueError(f"unknown noise mode {mode!r}")
        return mode == "numpy"

    def _require_n4(self, what: str):
        if self.n != 4:
            raise NotImplementedError(
                f"{what}: the CUDA path implements the n = 4 state [lon, lat, SOG, COG] "
                f"(this filter has n = {self.n}); only compute_weights / compute_sigma_points are dimension-generic"
            )

    def _resolve_process(self, non_linear_process):
        """-> (device model id, state dimension) of a process callable the CUDA path can run."""
        if non_linear_process is None:
            assert self.non_linear_process is not None, "Non-linear process is not set."
            non_linear_process = self.non_linear_process
        assert callable(non_linear_process), "Non-linear process model must be callable."
        if non_linear_process not in DEVICE_MODELS:
            raise NotImplementedError(
                "arbitrary Python callables cannot run inside a kernel; the CUDA path runs the process models of "
                "ship_track_estimators_b200.kalman_filters.non_linear_process: geodetic_dynamics (n = 4) and "
                "geodetic_dynamics_turn (n = 5)"
            )
        model, n = DEVICE_MODELS[non_linear_process]
        if n != self.n:
            raise ValueError(f"{non_linear_process.__name__} propagates {n} states, this filter has n = {self.n}")
        return model, n

    def _apply_measurement_model(self, z):
        """``z = self.measurement_model(z)`` (reference ``:221-225``) for the named models of
        :mod:`ship_track_estimators_b200.measurement_models`."""
        if self.measurement_model is None:
            return z
        assert callable(self.measurement_model), "Measurement model must be callable."
        from ..measurement_models import MEASUREMENT_MODELS

        if self.measurement_model not in MEASUREMENT_MODELS.values():
            raise NotImplementedError("measurement_model must be one of ship_track_estimators_b200.measurement_models."
                                      f"{sorted(MEASUREMENT_MODELS)} (arbitrary callables cannot be fused into the batched update)")
        return np.asarray(self.measurement_model(z), dtype=np.float64).reshape(-1, 1)

    def _model(self, P0=None):
        from ..batch import BatchedUKF

        return BatchedUKF(self.H, self.Q, self.R, self.P if P0 is None else P0, gating=self.gating,
                          measurement_model=self.measurement_model)

    def _step_problem(self, engine):
        from ..batch import TrackBatch  # noqa: F401  (keeps import order explicit)
        from .. import _native as nat

        p = nat.SteProblem()
        m = engine.model
        p.n_tracks, p.max_steps, p.max_obs, p.substeps, p.rate_repeat = 1, 1, 1, 1, 1
        p.flags = nat.STE_FLAG_GATING if m.gating else 0
        p.gate_max_iter, p.gate_chi, p.ld = int(m.gate_max_iter), float(m.gate_chi), 1
        for name, M in (("H", m.H), ("Q", m.Q), ("R", m.R), ("P0", m.P0)):
            getattr(p, name)[:] = M.reshape(-1).tolist()
        return p

    # ------------------------------------------------------------------ #
    # sigma points and weights (dimension-generic)                       #
    # ------------------------------------------------------------------ #
    def compute_weights(self, weight0: Optional[float] = None) -> np.ndarray:
        """Diagonal weight matrix, ``W0 = 1 - n/3`` by default (reference ``:109-142``)."""
        if weight0 is None:
            weight0 = 1 - self.n / 3.0
        assert weight0 < 1.0 and weight0 > -1.0, "Weight0 value ({}) is outside [-1, 1] range.".format(weight0)
        weightn = (1 - weight0) / (2 * self.n)
        np.fill_diagonal(self.weights, weightn)
        self.weights[0, 0] = weight0
        logging.debug("Weights\n\n%s", self.weights)
        return self.weights

    def compute_sigma_points(self, x: Optional[np.ndarray] = None, P: Optional[np.ndarray] = None) -> np.ndarray:
        """``X0 = x, Xi = x +/- sqrtm(n / (1 - W0) P)[:, i]`` (reference ``:76-107``), on the GPU."""
        import torch

        from .. import _native as nat

        if x is None:
            assert self.x is not None, "Set proper initial state estimate."
            x = self.x
        if P is None:
            assert self.P is not None, "Set proper initial state covariance matrix."
            P = self.P
        n = self.n
        if n > 8:
            raise NotImplementedError("sigma points on the CUDA path support n <= 8")
        scale = n / (1 - self.weights[0, 0])
        lib = nat.load()
        dev = torch.device("cuda")
        xd = torch.from_numpy(np.asarray(x, dtype=np.float64).reshape(n, 1).copy()).to(dev)
        Pd = torch.from_numpy(np.asarray(P, dtype=np.float64).reshape(n * n, 1).copy()).to(dev)
        Xd = torch.empty(n * self.n_sigma_points, 1, dtype=torch.float64, device=dev)
        st = torch.zeros(1, dtype=torch.int32, device=dev)
        nat.check(lib.ste_sigma_points_f64(n, 1, 1, float(scale), nat.ptr(xd), nat.ptr(Pd), nat.ptr(Xd), nat.ptr(st), nat.current_stream()))
        self.status |= int(st.item())
        self.sigma_points = Xd.cpu().numpy().reshape(n, self.n_sigma_points)
        return self.sigma_points

    # ------------------------------------------------------------------ #
    # single steps                                                       #
    # ------------------------------------------------------------------ #
    def predict(self, non_linear_process: Optional[Callable] = None, **non_linear_process_kwargs) -> None:
        """One unscented prediction (reference ``:144-207``); kwargs ``dt, c, sog_rate, cog_rate``."""
        import torch

        from .. import _native as nat

        model, _ = self._resolve_process(non_linear_process)
        if self.n != 4:
            return self._predict_generic(model, dict(non_linear_process_kwargs))
        kw = dict(non_linear_process_kwargs)
        if kw.get("c", None) is not None and np.size(kw["c"]) != 0:
            raise NotImplementedError("only c=None is supported (the reference never passes a control vector)")
        dt = float(kw["dt"])
        sog_rate, cog_rate = float(kw.get("sog_rate", 0.0)), float(kw.get("cog_rate", 0.0))
        self.x = self.x.reshape(-1, 1)
        self.compute_weights()
        engine = self._model()
        p = self._step_problem(engine)
        st = self._stages.get("predict")
        if st is None:
            st = self._stages["predict"] = _Stage([("x", 4), ("P", 16), ("dt", 1), ("sr", 1), ("cr", 1), ("noise", 4), ("status", 1),
                                                   ("sp0", 36), ("sp1", 36)])
        noisy = self._noise_on()
        st.put("x", self.x); st.put("P", self.P); st.put("dt", dt); st.put("sr", sog_rate); st.put("cr", cog_rate)
        st.put("noise", _unit_normals(1, 4) if noisy else np.zeros(4)); st.put("status", 0.0)
        st.upload("status")
        status_dev = st.dev_slot("status").view(torch.int32)
        nat.check(engine._lib.ste_ukf_predict_f64(
            C.byref(p), nat.ptr(st.dev_slot("x")), nat.ptr(st.dev_slot("P")), nat.ptr(st.dev_slot("dt")), nat.ptr(st.dev_slot("sr")),
            nat.ptr(st.dev_slot("cr")), nat.ptr(st.dev_slot("noise")) if noisy else None, nat.ptr(st.dev_slot("sp0")),
            nat.ptr(st.dev_slot("sp1")), nat.ptr(status_dev), nat.current_stream()))
        st.download()
        self.x = st.get("x").reshape(4, 1)
        self.P = st.get("P").reshape(4, 4)
        self.sigma_points_orig = st.get("sp0").reshape(4, 9)
        self.sigma_points = st.get("sp1").reshape(4, 9)
        self.status |= st.status()

    def _predict_generic(self, model, kw):
        """``predict`` for n != 4 through the dimension-generic kernel (``ste_ukf_predict_n_f64``)."""
        import torch

        from .. import _native as nat

        if kw.get("c", None) is not None and np.size(kw["c"]) != 0:
            raise NotImplementedError("only c=None is supported (the reference never passes a control vector)")
        n, L = self.n, self.n_sigma_points
        self.x = self.x.reshape(-1, 1)
        self.compute_weights()
        lib, dev = nat.load(), torch.device("cuda")
        f64 = dict(dtype=torch.float64, device=dev)
        up = lambda a, rows: torch.from_numpy(np.asarray(a, dtype=np.float64).reshape(rows, 1).copy()).to(dev)   # noqa: E731
        xd, Pd = up(self.x, n), up(self.P, n * n)
        scal = torch.tensor([[float(kw["dt"])], [float(kw.get("sog_rate", 0.0))], [float(kw.get("cog_rate", 0.0))]], **f64)
        noise = up(_unit_normals(1, n), n) if self._noise_on() else None
        sp0, sp1 = torch.empty(n * L, 1, **f64), torch.empty(n * L, 1, **f64)
        st = torch.zeros(1, dtype=torch.int32, device=dev)
        Q = np.ascontiguousarray(self.Q, dtype=np.float64)
        nat.check(lib.ste_ukf_predict_n_f64(n, model, 1, 1, Q.ctypes.data_as(C.POINTER(C.c_double)), nat.ptr(xd), nat.ptr(Pd), nat.ptr(scal[0]),
                                            nat.ptr(scal[1]), nat.ptr(scal[2]), nat.ptr(noise), nat.ptr(sp0), nat.ptr(sp1), nat.ptr(st),
                                            nat.current_stream()))
        self.x, self.P = xd.cpu().numpy().reshape(n, 1), Pd.cpu().numpy().reshape(n, n)
        self.sigma_points_orig, self.sigma_points = sp0.cpu().numpy().reshape(n, L), sp1.cpu().numpy().reshape(n, L)
        self.status |= int(st.item())

    def _update_generic(self, z):
        """``update`` for n != 4 through ``ste_ukf_update_n_f64`` (dense H and R, heading at index 3)."""
        import torch

        from .. import _native as nat

        if self.gating:
            raise NotImplementedError("the robustification is implemented for the n = 4 state")
        n = self.n
        lib, dev = nat.load(), torch.device("cuda")
        up = lambda a, rows: torch.from_numpy(np.asarray(a, dtype=np.float64).reshape(rows, 1).copy()).to(dev)   # noqa: E731
        xd, Pd, zd = up(self.x, n), up(self.P, n * n), up(z, n)
        noise = up(_unit_normals(1, n), n) if self._noise_on() else None
        st = torch.zeros(1, dtype=torch.int32, device=dev)
        H, R = (np.ascontiguousarray(M, dtype=np.float64) for M in (self.H, self.R))
        dp = C.POINTER(C.c_double)
        nat.check(lib.ste_ukf_update_n_f64(n, 1, 1, H.ctypes.data_as(dp), R.ctypes.data_as(dp), nat.ptr(xd), nat.ptr(Pd), nat.ptr(zd),
                                           nat.ptr(noise), nat.ptr(st), nat.current_stream()))
        self.x, self.P = xd.cpu().numpy().reshape(n, 1), Pd.cpu().numpy().reshape(n, n)
        self.status |= int(st.item())

    def _update_device(self, x, P, R, z, use_noise, gating=None):
        """Shared by ``update`` and ``check_robustness``: returns (x, P, iters, lambda, scale)."""
        import torch

        from ..batch import BatchedUKF
        from .. import _native as nat

        engine = BatchedUKF(self.H, self.Q, R, P, gating=self.gating if gating is None else gating)
        p = self._step_problem(engine)
        st = self._stages.get("update")
        if st is None:
            st = self._stages["update"] = _Stage([("x", 4), ("P", 16), ("z", 4), ("noise", 4), ("lam", 1), ("scale", 1), ("status", 1), ("iters", 1)])
        st.put("x", x); st.put("P", P); st.put("z", z); st.put("noise", _unit_normals(1, 4) if use_noise else np.zeros(4))
        st.put("lam", 1.0); st.put("scale", 1.0); st.put("status", 0.0); st.put("iters", 0.0)
        st.upload("iters")
        nat.check(engine._lib.ste_ukf_update_f64(
            C.byref(p), nat.ptr(st.dev_slot("x")), nat.ptr(st.dev_slot("P")), nat.ptr(st.dev_slot("z")),
            nat.ptr(st.dev_slot("noise")) if use_noise else None, nat.ptr(st.dev_slot("iters").view(torch.uint8)), nat.ptr(st.dev_slot("lam")),
            nat.ptr(st.dev_slot("scale")), nat.ptr(st.dev_slot("status").view(torch.int32)), nat.current_stream()))
        st.download()
        self.status |= st.status()
        a, _ = st.offsets["iters"]
        iters = int(st.host[a:a + 1].view(torch.uint8)[0])
        return st.get("x").reshape(4, 1), st.get("P").reshape(4, 4), iters, float(st.get("lam")[0]), float(st.get("scale")[0])

    def update(self, z: np.ndarray) -> None:
        """Linear measurement update with pseudo-inverse gain and Joseph-form covariance
        (reference ``:209-265``)."""
        z = self._apply_measurement_model(np.asarray(z, dtype=np.float64).reshape(-1, 1))
        if self.n != 4:
            return self._update_generic(z)
        if self.gating and self._noise_on():
            # the reference's own sequence (:228-236 with the robustification line enabled): the judging
            # loop draws fresh measurement noise per iteration, then the update draws once more with the
            # inflated R - a data-dependent number of draws, so the loop runs on the host around the
            # device evaluations of criterion_index / update_lambda_factor
            R = self.check_robustness(z, self.P, self.R)
            self.x, self.P, _, _, _ = self._update_device(self.x, self.P, R, z, True, gating=False)
            self.gate_iters.append(self.last_gate["iterations"])
            self.gate_lambda.append(self.last_gate["lambda_factor"])
            return
        self.x, self.P, it, lam, _ = self._update_device(self.x, self.P, self.R, z, self._noise_on())
        if self.gating:
            self.gate_iters.append(it)
            self.gate_lambda.append(lam)

    # ------------------------------------------------------------------ #
    # the two hot loops                                                  #
    # ------------------------------------------------------------------ #
    def _run_device(self, nsteps, dt, ship_track):
        from ..batch import TrackBatch, exact_update_mask

        self._resolve_process(None)
        if self.n != 4:
            return self._run_fleet_n(int(nsteps), dt, ship_track)
        N = int(nsteps)
        mask = exact_update_mask(dt, ship_track.dts, self.time)
        tape = None
        if self._noise_on():
            n_upd = 1 + int(mask.sum())
            meas = not self.gating
            draws = _unit_normals(N + (n_upd if meas else 0), 4)
            pred, upd, k = np.zeros((N, 4)), np.zeros((n_upd, 4)), 0
            if meas:
                upd[0] = draws[0]
                k = 1
            u = 1
            for s in range(N):  # reference call order: predict, then update when the step matches
                pred[s] = draws[k]
                k += 1
                if mask[s] and meas:
                    upd[u] = draws[k]
                    k += 1
                    u += 1
            tape = [dict(pred=pred, upd=upd)]
        engine = self._model()
        batch = TrackBatch.from_tracks([ship_track], [dt], x0=[np.asarray(self.x).reshape(-1)], time0=self.time,
                                       noise=tape, smoother=False)
        res = engine.run(batch, smoother=False)
        out = res.track(0)
        self.status |= out["status"]
        for s in range(N + 1):
            self.means.append(out["means"][s].reshape(4, 1).copy())
            self.covariances.append(out["covs"][s].copy())
        self.x = self.means[-1]
        self.P = self.covariances[-1]
        if N > 0:
            self.time = np.cumsum(np.concatenate(([np.float64(self.time)], dt)))[-1]
        ui = out["n_updates"] - 1
        self.c = np.asarray([ship_track.sog[ui], ship_track.cog[ui]]) if getattr(ship_track, "sog", None) is not None else None
        if self.gating:
            self.gate_iters.extend(out["gate_iters"].tolist())
            self.gate_lambda.extend(out["gate_lambda"].tolist())

    def _run_fleet_n(self, N, dt, ship_track):
        """``run`` at n = 5 (``geodetic_dynamics_turn``): one launch of the five-state fleet kernel on a tile of one
        track (``batch_n.BatchedUKFN``), bit-identical to the reference's time loop (``kalman_filter.py:76-111``)
        driven through ``predict`` / ``update``.  With ``noise="numpy"`` the same normals are drawn in the same
        order - n for the initial update, then per step n for the predict and n more when it updates - and
        replayed through the kernel's noise tapes."""
        from types import SimpleNamespace

        from ..batch import exact_update_mask
        from ..batch_n import BatchedUKFN, TrackBatchN

        n = self.n
        z = np.asarray(ship_track.z, dtype=np.float64)
        if z.shape[0] > n:
            raise ValueError("the measurement has more rows than the state")
        # the prior travels as a per-track P0: after a first run it is a filtered covariance, not exactly symmetric
        engine = BatchedUKFN(self.H, self.Q, self.R, measurement_model=self.measurement_model, gating=self.gating)
        track = SimpleNamespace(dts=ship_track.dts, z=np.concatenate([z, np.zeros((n - z.shape[0], z.shape[1]))]),
                                sog_rate=ship_track.sog_rate, cog_rate=ship_track.cog_rate)
        tape = None
        if self._noise_on():
            mask = exact_update_mask(dt, ship_track.dts, self.time)
            draws = _unit_normals(1 + N + int(mask.sum()), n)
            pred, upd = np.zeros((N, n)), [draws[0]]
            k = 1
            for s in range(N):   # reference call order: predict, then update when the step matches
                pred[s] = draws[k]
                k += 1
                if mask[s]:
                    upd.append(draws[k])
                    k += 1
            tape = [dict(pred=pred, upd=np.asarray(upd))]
        # IndexError past the last observation, as in the reference (:101-108)
        batch = TrackBatchN.from_tracks([track], [dt], x0=[np.asarray(self.x).reshape(-1)], time0=self.time, noise=tape,
                                        smoother=False, device="cuda", P0=[np.asarray(self.P, dtype=np.float64)])
        self.compute_weights()
        out = engine.run(batch, smoother=False).track(0)
        self.status |= out["status"]
        for s in range(N + 1):
            self.means.append(out["means"][s].reshape(n, 1).copy())
            self.covariances.append(out["covs"][s].copy())
        self.x = self.means[-1]
        self.P = self.covariances[-1]
        if N > 0:
            self.time = np.cumsum(np.concatenate(([np.float64(self.time)], dt)))[-1]

    def rts_step(self, fwd_means, fwd_vars, ship_track, *args, **kwargs):
        """Unscented RTS smoother over explicit filtered states (reference ``:267-351``).

        ``fwd_means (N+1, n, 1)``, ``fwd_vars (N+1, n, n)``; returns arrays of the same shapes (n = 4: the
        batched backward kernel on a tile of one track; other n: the dimension-generic kernel).
        Unlike the reference this does not overwrite ``ship_track.sog_rate / cog_rate`` with their
        ``np.repeat`` expansion (``:287-292``); the expansion is applied as an index map on the device.
        """
        import torch

        from ..batch import BatchedUKF, TrackBatch, TrackResults

        model, _ = self._resolve_process(None)
        fwd_means = np.asarray(fwd_means, dtype=np.float64)
        fwd_vars = np.asarray(fwd_vars, dtype=np.float64)
        if self.n != 4:
            return self._rts_generic(model, fwd_means, fwd_vars, ship_track)
        nstates = fwd_means.shape[0]
        N = nstates - 1
        if self.dt is None or len(self.dt) < N:
            raise IndexError("rts_step needs the dt array of the forward run (self.dt)")
        sog_rate = np.asarray(ship_track.sog_rate, dtype=np.float64)
        cog_rate = np.asarray(ship_track.cog_rate, dtype=np.float64)
        rep = int(nstates / len(ship_track.dts))
        if N > 0 and (rep < 1 or (N - 1) // rep >= min(len(sog_rate), len(cog_rate))):
            raise IndexError("index out of bounds for the repeated sog_rate / cog_rate arrays")
        dev = torch.device("cuda")

        def up(a):
            return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).to(dev)

        noise_bwd = None
        if self._noise_on() and N > 0:
            draws = _unit_normals(N, 4)  # drawn for step N-1 first
            noise_bwd = up(draws[::-1].reshape(N, 4, 1))
        m = len(sog_rate)
        batch = TrackBatch(
            x0=up(fwd_means[0].reshape(4, 1)), dt=up(np.asarray(self.dt, dtype=np.float64)[:N].reshape(N, 1) if N else np.zeros((1, 1))),
            sog_rate=up(sog_rate.reshape(m, 1)), cog_rate=up(cog_rate.reshape(m, 1)), z=[None] * 4,
            n_steps=torch.tensor([N], dtype=torch.int32, device=dev), rate_repeat_all=max(rep, 1),
            noise_bwd=noise_bwd, n_steps_host=np.array([N], dtype=np.int32),
        )
        engine = BatchedUKF(self.H, self.Q, self.R, self.P_orig)
        S = batch.max_steps + 1
        mean_f = torch.zeros(S, 4, 1, dtype=torch.float64, device=dev)
        cov_f = torch.zeros(S, 16, 1, dtype=torch.float64, device=dev)
        mean_f[:nstates] = up(fwd_means.reshape(nstates, 4, 1))
        cov_f[:nstates] = up(fwd_vars.reshape(nstates, 16, 1))
        res = TrackResults(
            mean_f=mean_f, cov_f=cov_f, mean_s=torch.empty_like(mean_f), cov_s=torch.empty_like(cov_f),
            status=torch.zeros(1, dtype=torch.int32, device=dev), n_updates=torch.zeros(1, dtype=torch.int32, device=dev),
            n_steps_host=batch.n_steps_host,
        )
        engine.backward(batch, res)
        self.status |= int(res.status.item())
        x = res.mean_s[:nstates].cpu().numpy().reshape(nstates, 4, 1)
        P = res.cov_s[:nstates].cpu().numpy().reshape(nstates, 4, 4)
        return x, P

    def _rts_generic(self, model, fwd_means, fwd_vars, ship_track):
        """``rts_step`` for n != 4: the whole backward loop in one launch of the dimension-generic kernel
        (``ste_urtss_backward_n_f64``), arithmetic written literally after the reference."""
        import torch

        from .. import _native as nat

        n, S = self.n, fwd_means.shape[0]
        N = S - 1
        if self.dt is None or len(self.dt) < N:
            raise IndexError("rts_step needs the dt array of the forward run (self.dt)")
        sog_rate = np.asarray(ship_track.sog_rate, dtype=np.float64).reshape(-1)
        cog_rate = np.asarray(ship_track.cog_rate, dtype=np.float64).reshape(-1)
        rep = int(S / len(ship_track.dts))
        m = min(len(sog_rate), len(cog_rate))
        if N > 0 and (rep < 1 or (N - 1) // rep >= m):
            raise IndexError("index out of bounds for the repeated sog_rate / cog_rate arrays")
        lib, dev = nat.load(), torch.device("cuda")
        up = lambda a, shape: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64).reshape(shape)).to(dev)   # noqa: E731
        mf, cf = up(fwd_means, (S, n, 1)), up(fwd_vars, (S, n * n, 1))
        ms, cs = torch.empty_like(mf), torch.empty_like(cf)
        dt = up(np.asarray(self.dt, dtype=np.float64)[:N] if N else np.zeros(1), (max(N, 1), 1))
        sr, cr = up(sog_rate[:m], (m, 1)), up(cog_rate[:m], (m, 1))
        noise = None
        if self._noise_on() and N > 0:
            noise = up(_unit_normals(N, n)[::-1], (N, n, 1))   # the reference draws for step N-1 first
        st = torch.zeros(1, dtype=torch.int32, device=dev)
        Q = np.ascontiguousarray(self.Q, dtype=np.float64)
        nat.check(lib.ste_urtss_backward_n_f64(n, model, 1, 1, S, max(rep, 1), m, Q.ctypes.data_as(C.POINTER(C.c_double)), nat.ptr(mf), nat.ptr(cf),
                                               nat.ptr(dt), nat.ptr(sr), nat.ptr(cr), nat.ptr(noise), nat.ptr(ms), nat.ptr(cs), nat.ptr(st),
                                               nat.current_stream()))
        self.status |= int(st.item())
        return ms.cpu().numpy().reshape(S, n, 1), cs.cpu().numpy().reshape(S, n, n)

    # ------------------------------------------------------------------ #
    # robustification (reference :353-511; dead code there)              #
    # ------------------------------------------------------------------ #
    def _gate_terms(self, z, P, R):
        """(gamma, denominator) of ``criterion_index`` / ``update_lambda_factor`` from the device."""
        import torch

        from ..batch import BatchedUKF
        from .. import _native as nat

        self._require_n4("criterion_index")
        engine = BatchedUKF(self.H, self.Q, R, P)
        p = self._step_problem(engine)
        dev = torch.device("cuda")
        up = lambda a, n: torch.from_numpy(np.asarray(a, dtype=np.float64).reshape(n, 1).copy()).to(dev)   # noqa: E731
        xd, Pd, zd = up(self.x, 4), up(P, 16), up(z, 4)
        out = torch.zeros(2, dtype=torch.float64, device=dev)
        nat.check(engine._lib.ste_gate_terms_f64(C.byref(p), nat.ptr(xd), nat.ptr(Pd), nat.ptr(zd), nat.ptr(out[0:1]), nat.ptr(out[1:2]),
                                                 nat.current_stream()))
        g, d = out.cpu().tolist()
        return g, d

    def criterion_index(self, z: np.ndarray, P: np.ndarray, R: np.ndarray) -> float:
        """Mahalanobis judging index ``|(z - x)^T pinv(H P H^T + R) (z - x)|`` (reference ``:389-428``;
        Chang, J Geod 88 (2014) 391-401, eq. 11/14)."""
        return self._gate_terms(z, P, R)[0]

    def update_lambda_factor(self, lambda_factor: float, criterion_index: float, chi_alpha: float, z: np.ndarray,
                             P: np.ndarray, R: np.ndarray) -> float:
        """``lambda + (gamma - chi) / ((z - x)^T S^+ R S^+ (z - x))`` (reference ``:430-483``, eq. 18)."""
        return lambda_factor + (criterion_index - chi_alpha) / self._gate_terms(z, P, R)[1]

    def check_robustness(self, z: np.ndarray, P: np.ndarray, R: np.ndarray) -> np.ndarray:
        """Mahalanobis-distance outlier judging: returns the inflated measurement covariance
        ``R * prod(lambda)`` (reference ``:353-387``).  With the noise off the whole loop is one
        kernel; with ``noise="numpy"`` it is the reference's loop, one fresh draw of measurement noise
        per evaluation (``:359-373``), around the device evaluations."""
        self._require_n4("check_robustness")
        if self._noise_on():
            z = np.asarray(z, dtype=np.float64).reshape(-1, 1)
            R = np.asarray(R, dtype=np.float64)
            lam, chi, it, scale = 1.0, 50.0, 0, 1.0
            draw = lambda: (np.random.normal(size=self.n) * np.sqrt(np.diag(R))).reshape(-1, 1)   # noqa: E731
            zn = z + draw()
            gamma = self.criterion_index(zn, P, R)
            while gamma > chi:
                zn = z + draw()
                lam = self.update_lambda_factor(lam, gamma, chi, zn, P, R)
                R = self.scale_measurement_uncertainty(R, lam)
                scale *= lam
                gamma = self.criterion_index(zn, P, R)
                it += 1
            self.last_gate = dict(iterations=it, lambda_factor=lam, scale=scale)
            return R
        keep = self.gating
        self.gating = True
        try:
            _, _, it, lam, scale = self._update_device(self.x, P, R, np.asarray(z, dtype=np.float64).reshape(-1, 1), False)
        finally:
            self.gating = keep
        self.last_gate = dict(iterations=it, lambda_factor=lam, scale=scale)
        return np.asarray(R) * scale

    def scale_measurement_uncertainty(self, R: np.ndarray, lambda_factor: float) -> np.ndarray:
        """``R * lambda`` (reference ``:484-511``)."""
        return R * lambda_factor
