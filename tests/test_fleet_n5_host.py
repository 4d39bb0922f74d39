"""CPU: the five-state fleet path's ABI surface and host-side packing, and the numpy oracle's five-state process.
No compute calls (no GPU): the invalid-argument paths return before any launch."""
import ctypes as C
import os
import subprocess
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest

from _helpers import GOLDEN, REPO

HEADER = os.path.join(REPO, "include", "ste_ukf.h")


def test_fleet_n_structs_match_c_layout():
    from ship_track_estimators_b200 import _native as nat

    structs = {"SteProblemN": nat.SteProblemN, "SteInputsN": nat.SteInputsN, "SteOutputsN": nat.SteOutputsN}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', "int main(void){"]
    for sname, cls in structs.items():
        lines.append(f'printf("{sname} %zu\\n", sizeof({sname}));')
        for fname, _ in cls._fields_:
            lines.append(f'printf("{sname}.{fname} %zu\\n", offsetof({sname}, {fname}));')
    lines.append("return 0;}")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "layout.c"), os.path.join(tmp, "layout")
        open(src, "w").write("\n".join(lines))
        subprocess.check_call(["gcc", "-std=c11", src, "-o", exe])
        out = subprocess.check_output([exe], text=True)
    c_layout = dict(line.split() for line in out.strip().splitlines())
    for sname, cls in structs.items():
        assert int(c_layout[sname]) == C.sizeof(cls), sname
        for fname, _ in cls._fields_:
            assert int(c_layout[f"{sname}.{fname}"]) == getattr(cls, fname).offset, f"{sname}.{fname}"


def _valid_problem(nat):
    p, i, o = nat.SteProblemN(), nat.SteInputsN(), nat.SteOutputsN()
    p.n, p.model, p.n_tracks, p.max_steps, p.max_obs, p.ld = 5, nat.STE_MODEL_GEODETIC_TURN, 4, 3, 2, 4
    for k in range(5):
        p.Q[k * 5 + k] = p.R[k * 5 + k] = p.P0[k * 5 + k] = 1.0
    fake = [0x1000 * (k + 1) for k in range(16)]   # never dereferenced: every case below fails validation
    i.x0, i.dt, i.upd_mask, i.sog_rate, i.rate_repeat = fake[:5]
    o.mean_f, o.cov_f, o.mean_s, o.cov_s, o.status = fake[5:10]
    return p, i, o


def test_fleet_n_invalid_arguments_without_a_launch(native_lib):
    from ship_track_estimators_b200 import _native as nat

    fwd, bwd = native_lib.ste_ukf_forward_n_f64, native_lib.ste_urtss_backward_tracks_n_f64
    call = lambda f, p, i, o: f(C.byref(p), C.byref(i), C.byref(o), None)   # noqa: E731
    p, i, o = _valid_problem(nat)
    p.n, p.model = 4, nat.STE_MODEL_GEODETIC
    assert call(fwd, p, i, o) == nat.STE_ERR_UNSUPPORTED and b"ste_ukf_forward_f64" in native_lib.ste_last_error()
    p.n, p.model = 5, nat.STE_MODEL_GEODETIC
    assert call(fwd, p, i, o) == nat.STE_ERR_UNSUPPORTED
    p, i, o = _valid_problem(nat)
    p.ld = 3   # ld < n_tracks
    assert call(fwd, p, i, o) == nat.STE_ERR_INVALID_ARG and b"ld" in native_lib.ste_last_error()
    p, i, o = _valid_problem(nat)
    p.max_obs = 0
    assert call(bwd, p, i, o) == nat.STE_ERR_INVALID_ARG
    for name in ("Q", "R", "P0"):
        p, i, o = _valid_problem(nat)
        getattr(p, name)[1] = 0.5   # asymmetric
        assert call(fwd, p, i, o) == nat.STE_ERR_UNSUPPORTED and b"symmetric" in native_lib.ste_last_error(), name
    p, i, o = _valid_problem(nat)
    i.upd_mask = None
    assert call(fwd, p, i, o) == nat.STE_ERR_INVALID_ARG and b"missing input" in native_lib.ste_last_error()
    p, i, o = _valid_problem(nat)
    i.rate_repeat = None
    assert call(bwd, p, i, o) == nat.STE_ERR_INVALID_ARG
    p, i, o = _valid_problem(nat)
    o.cov_s = None
    assert call(bwd, p, i, o) == nat.STE_ERR_INVALID_ARG and b"missing output" in native_lib.ste_last_error()
    p, i, o = _valid_problem(nat)
    o.mean_s = o.mean_f
    assert call(bwd, p, i, o) == nat.STE_ERR_INVALID_ARG and b"alias" in native_lib.ste_last_error()
    p, i, o = _valid_problem(nat)
    o.cov_s = o.cov_f
    assert call(fwd, p, i, o) == nat.STE_ERR_INVALID_ARG
    assert native_lib.ste_ukf_forward_n_f64(None, None, None, None) == nat.STE_ERR_INVALID_ARG


def _track(nobs, gaps, seed, rows=4):
    rng = np.random.default_rng(seed)
    return SimpleNamespace(dts=np.asarray(gaps, dtype=np.float64), z=rng.normal(size=(rows, nobs)), sog_rate=rng.normal(size=nobs),
                           cog_rate=rng.normal(size=nobs))


def test_track_batch_n_from_tracks_packing_on_the_host():
    from ship_track_estimators_b200.batch import exact_update_mask
    from ship_track_estimators_b200.batch_n import TrackBatchN
    from ship_track_estimators_b200.utils import generate_dts

    tracks = [_track(4, [1.0, 2.0, 1.0], 1), _track(6, [1.0] * 5, 2, rows=5), _track(3, [3.0, 3.0], 3)]
    ks = [1, 2, 3]
    dts = [generate_dts(t.dts, k) for t, k in zip(tracks, ks)]
    b = TrackBatchN.from_tracks(tracks, dts, device="cpu", smoother=True)
    b.check()
    lengths = [len(d) for d in dts]                        # 3, 10, 6
    assert list(b.order) == [1, 2, 0] and list(b.n_steps_host) == [10, 6, 3]
    assert b.max_steps == 10 and b.max_obs == 6 and len(b.z) == 5
    for col, i in enumerate(b.order):
        n, m, tr = lengths[i], tracks[i].z.shape[1], tracks[i]
        assert np.array_equal(b.dt[:n, col].numpy(), dts[i]) and not b.dt[n:, col].any()
        assert np.array_equal(b.upd_mask[:n, col].numpy().astype(bool), exact_update_mask(dts[i], tr.dts)) and not b.upd_mask[n:, col].any()
        zr = tr.z.shape[0]
        got = np.stack([r[:, col].numpy() for r in b.z])
        assert np.array_equal(got[:zr, :m], tr.z) and not got[zr:].any() and not got[:, m:].any()   # zero-padded to 5 rows
        assert np.array_equal(b.x0[:, col].numpy(), got[:, 0])
        assert np.array_equal(b.sog_rate[:m, col].numpy(), tr.sog_rate)
        assert int(b.rate_repeat[col]) == int((n + 1) / len(tr.dts))
    # the k = 3 grid does not re-sum to the fix times exactly everywhere: the mask comes from the reference's arithmetic
    col3 = list(b.order).index(2)
    assert b.upd_mask[:6, col3].numpy().tolist() == exact_update_mask(dts[2], tracks[2].dts).astype(np.uint8).tolist()
    unsorted = TrackBatchN.from_tracks(tracks, dts, device="cpu", sort_by_length=False)
    assert unsorted.order is None and list(unsorted.n_steps_host) == lengths
    noisy = TrackBatchN.from_tracks(tracks[:1], dts[:1], device="cpu", smoother=False, P0=[np.arange(25.0).reshape(5, 5)],
                                    noise=[dict(pred=np.ones((3, 5)), upd=2 * np.ones((2, 5)), bwd=None)])
    assert noisy.P0.shape == (25, 1) and noisy.P0[:, 0].tolist() == list(range(25))   # per-track prior, plane i*5+j, as given
    assert noisy.rate_repeat is None and noisy.noise_pred.shape == (3, 5, 1) and float(noisy.noise_upd[1].sum()) == 10.0
    assert float(noisy.noise_upd[2:].abs().sum()) == 0.0 and float(noisy.noise_bwd.abs().sum()) == 0.0
    # IndexError where the reference raises: more matched update times than observations, rates too short,
    # the smoother's rate index past the repeated arrays
    with pytest.raises(IndexError, match="update times matched"):
        TrackBatchN.from_tracks([_track(2, [1.0], 4)], [np.array([1.0, 0.0, 0.0])], device="cpu")
    short = _track(4, [1.0, 1.0, 1.0], 5)
    short.sog_rate = short.sog_rate[:2]
    with pytest.raises(IndexError, match="shorter"):
        TrackBatchN.from_tracks([short], [np.ones(3)], device="cpu")
    with pytest.raises(IndexError, match="rate index"):
        TrackBatchN.from_tracks([_track(4, [1.0, 1.0, 1.0], 6)], [np.array([3.0])], device="cpu", smoother=True)
    TrackBatchN.from_tracks([_track(4, [1.0, 1.0, 1.0], 6)], [np.array([3.0])], device="cpu", smoother=False)
    with pytest.raises(ValueError, match="rows"):
        TrackBatchN.from_tracks([_track(3, [1.0, 1.0], 7, rows=3)], [np.ones(2)], device="cpu")


def test_track_batch_n_check_rejects_wrong_shapes():
    import torch

    from ship_track_estimators_b200.batch_n import TrackBatchN

    b = TrackBatchN.from_tracks([_track(4, [1.0] * 3, 1), _track(3, [1.0] * 2, 2)], [np.ones(3), np.ones(2)], device="cpu")
    b.check()
    for name, bad in (("x0", torch.zeros(4, 2, dtype=torch.float64)), ("dt", torch.zeros(3, 3, dtype=torch.float64)),
                      ("upd_mask", torch.zeros(3, 2, dtype=torch.int32)), ("n_steps", torch.zeros(2, dtype=torch.int64)),
                      ("P0", torch.zeros(16, 2, dtype=torch.float64)), ("noise_pred", torch.zeros(3, 4, 2, dtype=torch.float64)),
                      ("rate_repeat", torch.ones(3, dtype=torch.int32)), ("cog_rate", torch.zeros(2, 4, dtype=torch.float64).t())):
        keep = getattr(b, name)
        setattr(b, name, bad)
        with pytest.raises(ValueError, match=name):
            b.check()
        setattr(b, name, keep)
    b.z = b.z[:4]
    with pytest.raises(ValueError, match="five observation rows"):
        b.check()


def test_oracle_reproduces_the_five_state_reference_tracks():
    import _oracle_n5 as O5

    d = np.load(os.path.join(GOLDEN, "kat_n5_tracks.npz"))
    for i in range(int(d["n"])):
        t = {k.split("_", 1)[1]: d[k] for k in d.files if k.startswith(f"t{i}_")}
        out = O5.run_track(t["x0"], d["P0"], d["H"], d["Q"], d["R"], t["dt_array"], t["dts"], t["z"], t["sog_rate"])
        for key in ("means", "means_s"):
            dm = out[key] - t[key]
            dm[:, 3] = (dm[:, 3] + 180.0) % 360.0 - 180.0
            assert float(np.max(np.abs(dm) / np.maximum(1.0, np.abs(t[key])))) <= 1e-12, (i, key)
        for key in ("covs", "covs_s"):
            assert max(float(np.max(np.abs(g - r)) / np.max(np.abs(r))) for g, r in zip(out[key], t[key])) <= 1e-12, (i, key)
