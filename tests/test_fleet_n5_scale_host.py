"""CPU: the five-state fleet path at scale without a GPU - the metrics entry point's ABI surface and argument checks,
fleet tiling, the host output buffers and estimate_fleet's settings validation."""
import ctypes as C
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest

from _helpers import REPO

HEADER = os.path.join(REPO, "include", "ste_ukf.h")
H5 = np.pad(np.eye(4), ((0, 1), (0, 1)))
E5 = np.eye(5)


def test_metrics_n_is_exported_with_the_header_abi(native_lib):
    from ship_track_estimators_b200 import _native as nat

    text = open(HEADER).read()
    assert int(re.search(r"#define STE_ABI_VERSION (\d+)", text).group(1)) == nat.STE_ABI_VERSION == native_lib.ste_version() == 7
    decl = re.search(r"int ste_track_metrics_n_f64\(([^;]*)\);", text).group(1)
    params = [p.strip() for p in decl.split(",")]
    assert params[:2] == ["const SteProblemN *prob", "const SteInputsN *in"] and len(params) == 9
    restype, argtypes = nat._PROTOTYPES["ste_track_metrics_n_f64"]
    assert restype is C.c_int and len(argtypes) == 9
    assert argtypes[0] == C.POINTER(nat.SteProblemN) and argtypes[1] == C.POINTER(nat.SteInputsN)
    assert all(a is nat._dptr for a in argtypes[2:8]) and argtypes[8] is C.c_void_p
    assert hasattr(native_lib, "ste_track_metrics_n_f64")


def _valid(nat):
    p, i = nat.SteProblemN(), nat.SteInputsN()
    p.n, p.model, p.n_tracks, p.max_steps, p.max_obs, p.ld = 5, nat.STE_MODEL_GEODETIC_TURN, 4, 3, 2, 4
    for k in range(5):
        p.Q[k * 5 + k] = p.R[k * 5 + k] = p.P0[k * 5 + k] = 1.0
    i.upd_mask = 0x1000   # never dereferenced: every case below returns before a launch
    out = [0x2000 * (k + 1) for k in range(6)]   # mean, rmse, cum_abs, max_abs, abs_diff, n_pairs
    return p, i, out


def test_metrics_n_invalid_arguments_without_a_launch(native_lib):
    from ship_track_estimators_b200 import _native as nat

    f = native_lib.ste_track_metrics_n_f64
    call = lambda p, i, out: f(p if p is None else C.byref(p), i if i is None else C.byref(i), *out, None)   # noqa: E731
    err = lambda: native_lib.ste_last_error()   # noqa: E731
    p, i, out = _valid(nat)
    assert call(None, i, out) == nat.STE_ERR_INVALID_ARG and call(p, None, out) == nat.STE_ERR_INVALID_ARG
    p.n, p.model = 4, nat.STE_MODEL_GEODETIC
    assert call(p, i, out) == nat.STE_ERR_UNSUPPORTED and b"ste_ukf_forward_f64" in err()
    p, i, out = _valid(nat)
    p.ld = 3
    assert call(p, i, out) == nat.STE_ERR_INVALID_ARG and b"ld" in err()
    p, i, out = _valid(nat)
    p.max_obs = 0
    assert call(p, i, out) == nat.STE_ERR_INVALID_ARG
    for name in ("Q", "R", "P0"):
        p, i, out = _valid(nat)
        getattr(p, name)[1] = 0.5
        assert call(p, i, out) == nat.STE_ERR_UNSUPPORTED and b"symmetric" in err(), name
    p, i, out = _valid(nat)
    i.upd_mask = None
    assert call(p, i, out) == nat.STE_ERR_INVALID_ARG and b"missing input" in err()
    p, i, out = _valid(nat)
    out[0] = None
    assert call(p, i, out) == nat.STE_ERR_INVALID_ARG and b"state array" in err()
    p, i, out = _valid(nat)   # every z row NULL: nothing to compare with
    assert call(p, i, out) == nat.STE_ERR_INVALID_ARG and b"observation row" in err()
    p.n_tracks = 0            # an empty tile launches nothing and succeeds
    assert call(p, i, out) == nat.STE_OK


def _track(nobs, seed):
    rng = np.random.default_rng(seed)
    return SimpleNamespace(dts=np.ones(nobs - 1), z=rng.normal(size=(4, nobs)), sog_rate=rng.normal(size=nobs), cog_rate=rng.normal(size=nobs))


def test_fleet_tiles_cut_as_plan_ragged_tiles_and_map_back():
    from ship_track_estimators_b200.batch_n import STATE_BUDGET, TrackBatchN, TrackResultsN
    from ship_track_estimators_b200.sharding import plan_ragged_tiles

    rng = np.random.default_rng(3)
    lengths = rng.integers(2, 40, size=57)
    tracks = [_track(int(m), k) for k, m in enumerate(lengths)]
    dts = [t.dts for t in tracks]
    budget, plan = 300, dict(granule=4, max_tracks=16)
    tiles = TrackBatchN.fleet_tiles(tracks, dts, device="cpu", state_budget=budget, **plan)
    order = np.argsort(-(lengths - 1), kind="stable")
    want = plan_ragged_tiles(lengths[order] - 1, budget, **plan)
    assert len(tiles) == len(want) > 2
    assert np.array_equal(np.concatenate([t.order for t in tiles]), order)
    for tile, (lo, hi) in zip(tiles, want):
        tile.check()
        assert tile.n_tracks == hi - lo and tile.max_steps == int(lengths[order[lo]]) - 1
        assert list(tile.n_steps_host) == list(lengths[order[lo:hi]] - 1)
        for j, i in enumerate(tile.order):   # column j holds the caller's track i
            m = int(lengths[i])
            assert np.array_equal(tile.z[0][:m, j].numpy(), tracks[i].z[0])
        # results of the tile answer to the caller's indices, and only to those it holds
        res = TrackResultsN(mean_f=tile.x0, cov_f=tile.x0, mean_s=None, cov_s=None, status=tile.n_steps, n_updates=tile.n_steps,
                            n_steps_host=tile.n_steps_host, order=tile.order)
        assert [res.column(int(i)) for i in tile.order] == list(range(tile.n_tracks))
        missing = next(i for i in range(len(tracks)) if i not in set(tile.order.tolist()))
        with pytest.raises(IndexError, match="not in this tile"):
            res.column(missing)
    assert STATE_BUDGET * 2 * 480 < 180e9 < 4e8 * 2 * 480   # two result sets of the default budget fit one B200
    one = TrackBatchN.fleet_tiles(tracks, dts, device="cpu")
    assert len(one) == 1 and np.array_equal(one[0].order, order)
    with pytest.raises(ValueError, match="empty"):
        TrackBatchN.fleet_tiles([], [], device="cpu")


def test_copy_from_and_input_bytes():
    from ship_track_estimators_b200.batch_n import TrackBatchN

    tracks = [_track(9, 1), _track(6, 2)]
    a = TrackBatchN.from_tracks(tracks, [t.dts for t in tracks], device="cpu")
    b = TrackBatchN.from_tracks(tracks[::-1], [t.dts[::-1].copy() for t in tracks[::-1]], device="cpu")
    assert a.input_bytes() == sum(t.numel() * t.element_size() for t in
                                  [a.x0, a.dt, a.upd_mask, a.n_steps, a.sog_rate, a.cog_rate, a.rate_repeat] + a.z)
    assert b.copy_from(a, non_blocking=False) and all(bool((x == y).all()) for x, y in zip(b.z, a.z))
    assert np.array_equal(b.order, a.order)
    c = TrackBatchN.from_tracks(tracks, [t.dts for t in tracks], device="cpu", smoother=False)
    assert not c.copy_from(a) and c.rate_repeat is None   # a different layout: nothing copied


def test_host_outputs_per_set(native_lib):
    import torch

    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks = [_track(9, 1), _track(6, 2), _track(4, 3)]
    b = TrackBatchN.from_tracks(tracks, [t.dts for t in tracks], device="cpu")
    T, S = 3, 9
    ukf = BatchedUKFN(H5, E5, E5, E5)
    want = {"all": {"mean_f": (S, 5, T), "cov_f": (S, 25, T), "mean_s": (S, 5, T), "cov_s": (S, 25, T)},
            "cli": {"mean_f": (S, 5, T), "diag_f": (S, 5, T), "mean_s": (S, 5, T), "diag_s": (S, 5, T)},
            "filtered": {"mean_f": (S, 5, T), "diag_f": (S, 5, T)}, "smoothed": {"mean_s": (S, 5, T), "diag_s": (S, 5, T)},
            "summary": {"final": (30, T), "metrics": (15, T)}}
    per_state = {"all": 480, "cli": 160, "filtered": 80, "smoothed": 80}
    assert set(ukf.OUTPUT_SETS) == set(want)
    for name, shapes in want.items():
        out = ukf.host_outputs(b, outputs=name, pinned=False)
        assert {k: tuple(v.shape) for k, v in out.items()} == {**shapes, "status": (T,), "n_updates": (T,)}, name
        assert out["status"].dtype == torch.int32 and all(v.dtype == torch.float64 for k, v in out.items() if k in shapes)
        if name in per_state:
            assert sum(v.numel() * 8 for k, v in out.items() if k in shapes) == per_state[name] * S * T
    with pytest.raises(ValueError, match="unknown output"):
        ukf.host_outputs(b, outputs=("mean_f", "turn"), pinned=False)
    for name in ("all", "cli", "smoothed"):
        with pytest.raises(ValueError, match="needs the smoother"):
            ukf.host_outputs(b, outputs=name, smoother=False, pinned=False)
    assert set(ukf.host_outputs(b, outputs="filtered", smoother=False, pinned=False)) == {"mean_f", "diag_f", "status", "n_updates"}
    with pytest.raises(KeyError):
        ukf.host_outputs(b, outputs="everything", pinned=False)


@pytest.mark.parametrize("dim", [3, 5, 6])
def test_estimate_fleet_settings(dim, tmp_path, monkeypatch):
    """dim 3 and 6 raise before the file is read; dim 5 is accepted and goes on to read it (here: a missing file)."""
    from ship_track_estimators_b200.cli import writers

    settings = {"dim": dim, "H": [1.0] * dim, "R": [1e-3] * dim, "Q": [1e-2] * dim, "P": [1.0] * dim, "dt": -1, "nsteps": 1}
    missing = str(tmp_path / "no_such.csv")
    if dim == 5:
        with pytest.raises(FileNotFoundError):
            writers.estimate_fleet(missing, settings, device="cpu")
        bad = dict(settings, H=[1.0] * 4)   # 4 entries for a 5-state model
        with pytest.raises(AssertionError, match="Dimension mismatch"):
            writers.estimate_fleet(missing, bad, device="cpu")
        from test_host_dropin import _fleet_csv

        csv = str(tmp_path / "fleet.csv")
        _fleet_csv(csv, seed=5, n_ships=6, time_ordered=True)   # every ship has fewer than 40 fixes
        with pytest.raises(ValueError, match="enough fixes"):
            writers.estimate_fleet(csv, settings, id_col="primary.id", device="cpu", min_fixes=40)
    else:
        with pytest.raises(NotImplementedError, match="4-state"):
            writers.estimate_fleet(missing, settings, device="cpu")
