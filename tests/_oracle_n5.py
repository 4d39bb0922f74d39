"""Five-state (turn-rate) restatement of the reference's UKF + URTSS loops for the tests of the fleet path.

The state is ``[lon, lat, SOG, COG, COG rate]``; the process is the geodetic step with the turn rate taken from the
state, where it persists (the model ``tests/golden/make_n4_golden.py`` builds from the reference's own
``geodetic_dynamics``).  The loops below restate ``oracle.ukf_numpy.predict`` / ``run_forward`` / ``run_smoother``
(reference ``kalman_filter.py:36-117``, ``unscented.py:144-351``) line for line with that process; the building blocks
- sigma points, weights, the linear update, the update mask, the angle wrap - are the oracle's own.
Test infrastructure: the product package never imports it.
"""
from __future__ import annotations

import warnings

import numpy as np

from oracle import ukf_numpy as O


def geodetic_dynamics_turn(x, dt, sog_rate=0.0, cog_rate=0.0):
    """The geodetic step with the turn rate taken from state 4 (``cog_rate`` is ignored); the turn rate persists."""
    return np.concatenate([O.geodetic_dynamics(x[:4], dt, sog_rate, x[4]), x[4:5]])


def predict(x, P, Q, dt, sog_rate):
    """kalman_filters/unscented.py:144-207 with the five-state process and zero noise.  Returns (x, P)."""
    n = x.shape[0]
    w0, wi = O.ut_weights(n)
    X = O.sigma_points(x, P, w0)
    Y = np.empty_like(X)
    for j in range(X.shape[1]):
        Y[:, j] = geodetic_dynamics_turn(X[:, j], dt, sog_rate)
    w = np.full(X.shape[1], wi)
    w[0] = w0
    mean = (Y * w).sum(axis=1)  # :195
    dev = Y - mean[:, None]  # :205
    return mean, O._weighted_outer(dev, dev, w0, wi) + Q


def run_forward(x0, P0, H, Q, R, dt_array, dts, z, sog_rate):
    """kalman_filter.py:36-117.  Returns dict(means (N+1, 5), covs (N+1, 5, 5)); index 0 is the prior."""
    noise = O.ZeroNoise()
    x = np.asarray(x0, dtype=np.float64).reshape(-1).copy()
    P = np.asarray(P0, dtype=np.float64).copy()
    mask = O.update_mask(dt_array, dts)
    means, covs = [x.copy()], [P.copy()]
    ui = 0
    x, P = O.update(x, P, H, R, z[:, ui].copy(), noise)  # :81
    for step, dt in enumerate(dt_array):
        x, P = predict(x, P, Q, dt, sog_rate[ui])  # :90-95
        if mask[step]:  # :101
            ui += 1
            x, P = O.update(x, P, H, R, z[:, ui].copy(), noise)
        means.append(x.copy())
        covs.append(P.copy())
    return dict(means=np.asarray(means), covs=np.asarray(covs))


def run_smoother(means, covs, Q, dt_array, n_dts, sog_rate):
    """unscented.py:267-351 with the five-state process and zero noise (P_b about the filtered mean, pinv gain)."""
    xs = np.array(means, dtype=np.float64, copy=True)
    Ps = np.array(covs, dtype=np.float64, copy=True)
    nstates, n = xs.shape
    sog_rep = np.repeat(np.asarray(sog_rate, dtype=np.float64), O.rts_rate_index(nstates, n_dts))
    w0, wi = O.ut_weights(n)
    for step in range(nstates - 2, -1, -1):
        X = O.sigma_points(xs[step], Ps[step], w0)
        Y = np.empty_like(X)
        for j in range(X.shape[1]):
            Y[:, j] = geodetic_dynamics_turn(X[:, j], dt_array[step], sog_rep[step])
        w = np.full(X.shape[1], wi)
        w[0] = w0
        x_b = (Y * w).sum(axis=1)
        dev_f = Y - xs[step][:, None]
        P_b = O._weighted_outer(dev_f, dev_f, w0, wi) + Q  # :324-325
        D = O._weighted_outer(X - xs[step][:, None], Y - x_b[:, None], w0, wi)  # :328-330
        K = D @ np.linalg.pinv(P_b)  # :333
        y = xs[step + 1] - x_b
        y[3] = O.wrap180(y[3])  # :340
        xs[step] = xs[step] + K @ y
        xs[step][3] = xs[step][3] % 360.0  # :346
        Ps[step] = Ps[step] + (K @ (Ps[step + 1] - P_b)) @ K.T  # :349
    return xs, Ps


def run_track(x0, P0, H, Q, R, dt_array, dts, z, sog_rate):
    """Forward + backward for one five-state track."""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = run_forward(x0, P0, H, Q, R, dt_array, dts, z, sog_rate)
        out["means_s"], out["covs_s"] = run_smoother(out["means"], out["covs"], Q, dt_array, len(dts), sog_rate)
    return out
