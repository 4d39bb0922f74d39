"""GPU: the five-state fleet path (``batch_n``: ``ste_ukf_forward_n_f64`` / ``ste_urtss_backward_tracks_n_f64``) against
the reference's known answers, bit for bit against the single-step n = 5 kernels, at size against the numpy oracle, and
against the n = 4 batched path with an inert turn rate."""
import ctypes as C
import os
from types import SimpleNamespace

import numpy as np
import pytest

from _helpers import GOLDEN, TOL, circ_diff

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True, scope="module")
def _release_cached_blocks():
    """Hand the cached device blocks of this module's tiles back when it ends, so that the modules after it start
    from the allocator state they would see without it."""
    yield
    import torch

    if torch.cuda.is_available():
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


H5 = np.zeros((5, 5))
H5[:4, :4] = np.eye(4)
Q5 = np.diag([1e-2, 1e-2, 1e-4, 1e-4, 1e-5])
R5 = np.diag([1e-3, 1e-3, 0.5, 4.0, 0.0])
P5 = np.diag([1.0, 1.0, 1.0, 4.0, 1e-2])


def _errs(got_m, got_c, ref_m, ref_c):
    """(mean, cov) errors as test_gpu_golden's n = 5 run test measures them."""
    dm = np.asarray(got_m).reshape(ref_m.shape) - ref_m
    dm[:, 3] = circ_diff(np.asarray(got_m)[:, 3], ref_m[:, 3])
    em = float(np.max(np.abs(dm) / np.maximum(1.0, np.abs(ref_m))))
    ec = max(float(np.max(np.abs(g - r)) / np.max(np.abs(r))) for g, r in zip(np.asarray(got_c), ref_c))
    return em, ec


def _fleet(T, nobs_max, seed, ks=(1, 2, 3), nobs_min=3, dts_choices=(1.0, 2.0, 3.0)):
    """Ragged five-state tracks (all five observation rows; the turn rate starts non-zero) with their step grids."""
    from ship_track_estimators_b200.synthetic import make_tracks
    from ship_track_estimators_b200.utils import generate_dts

    syn = make_tracks(T, nobs_max, seed=seed, device="cpu", nobs_min=nobs_min, dts_choices=dts_choices)
    rng = np.random.default_rng(seed)
    tracks, dts, x0 = [], [], []
    for t in range(T):
        m = int(syn.nobs[t])
        z = np.stack([syn.lon[:m, t].numpy(), syn.lat[:m, t].numpy(), syn.sog[:m, t].numpy(), syn.cog[:m, t].numpy(),
                      rng.normal(size=m) * 0.2])
        tr = SimpleNamespace(dts=syn.dts[: m - 1, t].numpy().copy(), z=z, sog_rate=syn.sog_rate[:m, t].numpy().copy(),
                             cog_rate=syn.cog_rate[:m, t].numpy().copy())
        tracks.append(tr)
        dts.append(generate_dts(tr.dts, ks[t % len(ks)]))
        x0.append(np.append(z[:4, 0], 0.3 * rng.normal()))
    return tracks, dts, x0


def test_reference_tracks_through_one_tile(cuda, native_lib):
    """The three reference tracks of kat_n5_tracks.npz (k = 1, 2, 2) through ONE BatchedUKFN.run tile."""
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    d = np.load(os.path.join(GOLDEN, "kat_n5_tracks.npz"))
    ts = [{k.split("_", 1)[1]: d[k] for k in d.files if k.startswith(f"t{i}_")} for i in range(int(d["n"]))]
    tracks = [SimpleNamespace(dts=t["dts"], z=t["z"], sog_rate=t["sog_rate"], cog_rate=t["cog_rate"]) for t in ts]
    b = TrackBatchN.from_tracks(tracks, [t["dt_array"] for t in ts], x0=[t["x0"] for t in ts], device=cuda)
    res = BatchedUKFN(d["H"], d["Q"], d["R"], d["P0"]).run(b)
    res.check_status()
    for i, t in enumerate(ts):
        out = res.track(i)
        em, ec = _errs(out["means"], out["covs"], t["means"], t["covs"])
        es, ecs = _errs(out["means_s"], out["covs_s"], t["means_s"], t["covs_s"])
        print(f"  n = 5 fleet track {i}: filtered {em:.1e} {ec:.1e}  smoothed {es:.1e} {ecs:.1e}")
        assert out["means"].shape == t["means"].shape and max(em, ec, es, ecs) <= TOL, (i, em, ec, es, ecs)
        assert out["status"] == 0 and out["n_updates"] == t["z"].shape[1]


def _single_step_reference(tracks, dts, x0, noise, dev):
    """Every track filtered step by step through ste_ukf_predict_n_f64 / ste_ukf_update_n_f64, then smoothed alone by
    ste_urtss_backward_n_f64: the class API's kernels.  Tracks in decreasing length, so the active ones are a prefix;
    the updates of a step run on the tracks gathered into a tile of their own."""
    import torch

    from ship_track_estimators_b200 import _native as nat
    from ship_track_estimators_b200.batch import exact_update_mask

    lib, f64 = nat.load(), dict(dtype=torch.float64, device=dev)
    dp = C.POINTER(C.c_double)
    Qc, Hc, Rc = (np.ascontiguousarray(M) for M in (Q5, H5, R5))
    T = len(tracks)
    lens = [len(d) for d in dts]
    assert lens == sorted(lens, reverse=True)
    N = lens[0]
    x = torch.tensor(np.stack(x0, axis=1), **f64).contiguous()
    P = torch.tensor(np.repeat(P5.reshape(25, 1), T, axis=1), **f64).contiguous()
    means, covs = [[x[:, t].cpu().numpy()] for t in range(T)], [[P[:, t].cpu().numpy().reshape(5, 5)] for t in range(T)]
    masks = [exact_update_mask(dts[t], tracks[t].dts) for t in range(T)]
    ui = np.zeros(T, dtype=np.int64)

    def update(cols, u_idx):
        k = len(cols)
        idx = torch.tensor(cols, device=dev)
        xs, Ps = x[:, idx].contiguous(), P[:, idx].contiguous()
        z = torch.tensor(np.stack([tracks[t].z[:, u] for t, u in zip(cols, u_idx)], axis=1), **f64).contiguous()
        nz = None
        if noise is not None:
            nz = torch.tensor(np.stack([noise[t]["upd"][u] for t, u in zip(cols, u_idx)], axis=1), **f64).contiguous()
        nat.check(lib.ste_ukf_update_n_f64(5, k, k, Hc.ctypes.data_as(dp), Rc.ctypes.data_as(dp), nat.ptr(xs), nat.ptr(Ps), nat.ptr(z),
                                           nat.ptr(nz), None, nat.current_stream()))
        x[:, idx], P[:, idx] = xs, Ps

    update(list(range(T)), [0] * T)
    for s in range(N):
        act = sum(1 for n in lens if n > s)
        xa, Pa = x[:, :act].contiguous(), P[:, :act].contiguous()   # ld = act: a contiguous prefix tile
        dt = torch.tensor([dts[t][s] for t in range(act)], **f64)
        sr = torch.tensor([tracks[t].sog_rate[ui[t]] for t in range(act)], **f64)
        cr = torch.tensor([tracks[t].cog_rate[ui[t]] for t in range(act)], **f64)
        nz = None if noise is None else torch.tensor(np.stack([noise[t]["pred"][s] for t in range(act)], axis=1), **f64).contiguous()
        nat.check(lib.ste_ukf_predict_n_f64(5, nat.STE_MODEL_GEODETIC_TURN, act, act, Qc.ctypes.data_as(dp), nat.ptr(xa), nat.ptr(Pa),
                                            nat.ptr(dt), nat.ptr(sr), nat.ptr(cr), nat.ptr(nz), None, None, None, nat.current_stream()))
        x[:, :act], P[:, :act] = xa, Pa
        upd = [t for t in range(act) if masks[t][s]]
        for t in upd:
            ui[t] += 1
        if upd:
            update(upd, [int(ui[t]) for t in upd])
        xh, Ph = x[:, :act].cpu().numpy(), P[:, :act].cpu().numpy()
        for t in range(act):
            means[t].append(xh[:, t].copy())
            covs[t].append(Ph[:, t].reshape(5, 5).copy())
    out = []
    for t in range(T):
        S, m = lens[t] + 1, tracks[t].z.shape[1]
        mf = torch.tensor(np.stack(means[t]).reshape(S, 5, 1), **f64)
        cf = torch.tensor(np.stack(covs[t]).reshape(S, 25, 1), **f64)
        ms, cs = torch.empty_like(mf), torch.empty_like(cf)
        dt = torch.tensor(np.asarray(dts[t]).reshape(-1, 1) if lens[t] else np.zeros((1, 1)), **f64)
        sr, cr = (torch.tensor(np.asarray(a[:m]).reshape(m, 1), **f64) for a in (tracks[t].sog_rate, tracks[t].cog_rate))
        nb = None if noise is None else torch.tensor(noise[t]["bwd"].reshape(-1, 5, 1), **f64).contiguous()
        rep = int(S / len(tracks[t].dts))
        nat.check(lib.ste_urtss_backward_n_f64(5, nat.STE_MODEL_GEODETIC_TURN, 1, 1, S, rep, m, Qc.ctypes.data_as(dp), nat.ptr(mf), nat.ptr(cf),
                                               nat.ptr(dt), nat.ptr(sr), nat.ptr(cr), nat.ptr(nb), nat.ptr(ms), nat.ptr(cs), None,
                                               nat.current_stream()))
        out.append(dict(means=np.stack(means[t]), covs=np.stack(covs[t]), means_s=ms.cpu().numpy().reshape(S, 5),
                        covs_s=cs.cpu().numpy().reshape(S, 5, 5)))
    return out


def test_bit_identical_to_the_single_step_kernels(cuda, native_lib):
    """A ragged tile of 64 tracks (5-200 steps, k in {1, 2, 3}, every covariance entry excited by a full prior and five
    observed rows), with zero noise and with all three tapes: every track's filtered and smoothed states equal the
    single-step kernels driven step by step, and the smoother on that track alone."""
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(64, 67, seed=11, nobs_min=6)
    order = np.argsort([-len(d) for d in dts], kind="stable")
    tracks, dts, x0 = [tracks[j] for j in order], [dts[j] for j in order], [x0[j] for j in order]
    lens = [len(d) for d in dts]
    assert min(lens) >= 5 and max(lens) <= 200 and max(lens) >= 100
    rng = np.random.default_rng(3)
    tapes = [dict(pred=rng.normal(size=(n, 5)), upd=rng.normal(size=(tr.z.shape[1], 5)), bwd=rng.normal(size=(n, 5)))
             for tr, n in zip(tracks, lens)]
    engine = BatchedUKFN(H5, Q5, R5, P5)
    for noise in (None, tapes):
        b = TrackBatchN.from_tracks(tracks, dts, x0=x0, noise=noise, device=cuda)
        res = engine.run(b).to_host()
        ref = _single_step_reference(tracks, dts, x0, noise, cuda)
        for i, r in enumerate(ref):
            got = res.track(i)
            assert np.count_nonzero(got["covs"][-1]) == 25
            for key in ("means", "covs", "means_s", "covs_s"):
                assert np.array_equal(got[key], r[key]), (noise is not None, i, key)


def test_at_size_against_the_numpy_oracle(cuda, native_lib):
    """256 ragged tracks, up to 300 steps, gaps of 1-3 h, k <= 2, against the n = 5 numpy oracle at 1e-9."""
    import _oracle_n5 as O5
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, x0 = _fleet(256, 151, seed=29, ks=(1, 2), nobs_min=20)
    res = BatchedUKFN(H5, Q5, R5, P5).run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda)).to_host()
    res.check_status()
    worst = np.zeros(4)
    for i, (tr, dt) in enumerate(zip(tracks, dts)):
        ref = O5.run_track(x0[i], P5, H5, Q5, R5, dt, tr.dts, tr.z, tr.sog_rate)
        got = res.track(i)
        e = _errs(got["means"], got["covs"], ref["means"], ref["covs"]) + _errs(got["means_s"], got["covs_s"], ref["means_s"], ref["covs_s"])
        worst = np.fmax(worst, e)
        assert max(e) <= TOL, (i, e)
    print(f"  n = 5 fleet vs numpy oracle, worst (filtered mean, cov, smoothed mean, cov): {worst}")


def test_inert_turn_rate_matches_the_n4_batched_path(cuda, native_lib):
    """Zero prior variance and zero Q on the turn rate, cog_rate = 0 on the n = 4 side: the first four states of a ragged
    n = 5 tile match BatchedUKF.run at n = 4 within 1e-8 (the n = 5 transform with an inert fifth state IS the n = 4
    one: the scale n / (1 - W0) = 3 and Wi = 1/6 are the same and the two extra sigma points sit on the mean)."""
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tracks, dts, _ = _fleet(48, 40, seed=17, ks=(1, 2), nobs_min=8, dts_choices=(1.0, 2.0))
    for tr in tracks:
        tr.cog_rate = np.zeros_like(tr.cog_rate)
        tr.z = tr.z[:4]
    H4, Q4, R4, P4 = np.diag([1.0, 1, 0, 0]), np.diag([1e-2, 1e-2, 1e-4, 1e-4]), np.diag([1e-3, 1e-3, 0, 0]), np.eye(4)
    pad = lambda M: np.pad(M, ((0, 1), (0, 1)))   # noqa: E731
    r4 = BatchedUKF(H4, Q4, R4, P4).run(TrackBatch.from_tracks(tracks, dts, device=cuda)).to_host()
    r5 = BatchedUKFN(pad(H4), pad(Q4), pad(R4), pad(P4)).run(TrackBatchN.from_tracks(tracks, dts, device=cuda)).to_host()
    for i in range(len(tracks)):
        a, b = r4.track(i), r5.track(i)
        for mk, ck in (("means", "covs"), ("means_s", "covs_s")):
            assert np.all(b[mk][:, 4] == 0.0) and np.all(b[ck][:, 4, :] == 0.0)
            em, ec = _errs(b[mk][:, :4], b[ck][:, :4, :4], a[mk], a[ck])
            assert em <= 1e-8 and ec <= 1e-8, (i, mk, em, ec)


def test_packing_composition_determinism_and_device_ingest(cuda, native_lib, tmp_path):
    """sort_by_length on / off, a track alone vs inside the tile and two runs: bit-identical.  from_batch of a
    device-ingested fleet (cadence form, k = 2) equals from_tracks fed the same inputs read back from the n = 4 tile."""
    import torch

    from test_host_dropin import _fleet_csv
    from ship_track_estimators_b200.batch import exact_update_mask
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.ingest import DeviceFleetFixes, read_csv_fleet_device

    tracks, dts, x0 = _fleet(40, 30, seed=5)
    engine = BatchedUKFN(H5, Q5, R5, P5)
    a = engine.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda)).to_host()
    b = engine.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda, sort_by_length=False)).to_host()
    c = engine.run(TrackBatchN.from_tracks(tracks, dts, x0=x0, device=cuda)).to_host()
    assert a.order is not None and b.order is None
    for i in range(len(tracks)):
        alone = engine.run(TrackBatchN.from_tracks([tracks[i]], [dts[i]], x0=[x0[i]], device=cuda)).track(0) if i % 7 == 0 else None
        ta, tb, tc = a.track(i), b.track(i), c.track(i)
        for key in ("means", "covs", "means_s", "covs_s"):
            assert np.array_equal(ta[key], tb[key]) and np.array_equal(ta[key], tc[key]), (i, key)
            if alone is not None:
                assert np.array_equal(ta[key], alone[key]), (i, key)

    csv = str(tmp_path / "fleet.csv")
    _fleet_csv(csv, seed=21, n_ships=14, string_labels=False, time_ordered=True)
    f = read_csv_fleet_device(csv, id_col="primary.id", device=cuda)
    # ships with a single fix cannot be filtered, and the cadence form needs strictly positive gaps
    valid = torch.arange(f.dts.shape[0], device=cuda)[:, None] < (f.n_obs.to(torch.int64) - 1)[None, :]
    keep = torch.nonzero((f.n_obs >= 2) & ((f.dts > 0) | ~valid).all(dim=0)).flatten()
    assert len(keep) >= 4
    f = DeviceFleetFixes([f.ids[i] for i in keep.tolist()], f.lon[:, keep].contiguous(), f.lat[:, keep].contiguous(),
                         f.dts[:, keep].contiguous(), f.n_obs[keep].contiguous(), f.stats)
    b4 = f.to_batch(substeps=2)
    bn = TrackBatchN.from_batch(b4, turn_rate0=0.1)
    assert bn.x0.shape[0] == 5 and bn.z[4] is None and bn.dt is b4.dt
    got = engine.run(bn).to_host()
    k, T = 2, b4.n_tracks
    nsteps = b4.n_steps.cpu().numpy() if b4.n_steps is not None else np.full(T, b4.max_steps)
    cols = []
    for j in range(T):
        n = int(nsteps[j])
        dt = b4.dt[:n, j].cpu().numpy()
        m = n // k + 1
        z = np.stack([np.zeros(m) if r is None else r[:m, j].cpu().numpy() for r in b4.z])
        tr = SimpleNamespace(dts=dt.reshape(-1, k).sum(axis=1), z=z, sog_rate=b4.sog_rate[:m, j].cpu().numpy(),
                             cog_rate=b4.cog_rate[:m, j].cpu().numpy())
        assert np.array_equal(bn.upd_mask[:n, j].cpu().numpy().astype(bool), exact_update_mask(dt, tr.dts))
        cols.append((tr, dt, np.append(b4.x0[:, j].cpu().numpy(), 0.1)))
    ref = engine.run(TrackBatchN.from_tracks([c_[0] for c_ in cols], [c_[1] for c_ in cols], x0=[c_[2] for c_ in cols],
                                             device=cuda, sort_by_length=False)).to_host()
    for j in range(T):
        n = int(nsteps[j])
        for key in ("mean_f", "cov_f", "mean_s", "cov_s"):
            assert torch.equal(getattr(got, key)[: n + 1, :, j], getattr(ref, key)[: n + 1, :, j]), (j, key)


def test_status_overrun_and_stale_results(cuda, native_lib):
    """A hand-built tile whose mask matches more steps than it has observations sets STE_STATUS_OBS_OVERRUN (the update is
    skipped) and check_status raises; results filtered from one tile are refused by the smoother of another."""
    import torch

    from ship_track_estimators_b200 import _native as nat
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    T, N, M = 3, 6, 3
    f64 = dict(dtype=torch.float64, device=cuda)
    b = TrackBatchN(x0=torch.tensor([[10.0] * T, [50.0] * T, [12.0] * T, [90.0] * T, [0.1] * T], **f64), dt=torch.ones(N, T, **f64),
                    upd_mask=torch.ones(N, T, dtype=torch.uint8, device=cuda), n_steps=torch.tensor([6, 2, 1], dtype=torch.int32, device=cuda),
                    sog_rate=torch.zeros(M, T, **f64), cog_rate=None, z=[torch.full((M, T), v, **f64) for v in (10.0, 50.0, 12.0, 90.0)] + [None],
                    rate_repeat=torch.ones(T, dtype=torch.int32, device=cuda), n_steps_host=np.array([6, 2, 1]))
    engine = BatchedUKFN(H5, Q5, R5, P5)
    res = engine.run(b)
    st = res.status.cpu().numpy()
    assert st[0] & nat.STE_STATUS_OBS_OVERRUN and not st[1] & nat.STE_STATUS_OBS_OVERRUN and not st[2]
    assert res.n_updates.cpu().tolist() == [3, 3, 2]
    with pytest.raises(IndexError, match="matched more update times"):
        res.check_status()
    assert res.check_status(raise_on=0)["obs_overrun"] == 1
    other = TrackBatchN(**{**b.__dict__})
    with pytest.raises(ValueError, match="different tile"):
        engine.backward(other, res)
    with pytest.raises(ValueError, match="BatchedUKF"):
        from ship_track_estimators_b200.kalman_filters import geodetic_dynamics

        BatchedUKFN(H5, Q5, R5, P5, process=geodetic_dynamics)
    with pytest.raises(NotImplementedError):
        BatchedUKFN(H5, Q5, R5, P5, gating=True)


def test_class_run_equals_public_steps_under_seeded_numpy_noise(cuda, native_lib):
    """The class API at n = 5 with noise="numpy": ``run`` (one fleet launch) equals, bit for bit, the same filter driven
    through the public ``update`` / ``predict`` calls with the same seed; results accumulate across calls."""
    from ship_track_estimators_b200.batch import exact_update_mask
    from ship_track_estimators_b200.kalman_filters import UnscentedKalmanFilter, geodetic_dynamics_turn
    from ship_track_estimators_b200.measurement_models import wrap_course

    tracks, dts, x0 = _fleet(2, 25, seed=41, ks=(2, 3), nobs_min=20)
    tr, dt = tracks[1], dts[1]
    tr.z = tr.z[:4]
    make = lambda: UnscentedKalmanFilter(H=H5, Q=Q5, R=R5, P=P5, x0=x0[1], non_linear_process=geodetic_dynamics_turn,   # noqa: E731
                                         measurement_model=wrap_course, noise="numpy")
    np.random.seed(1234)
    u1 = make()
    m1, c1 = u1.run(len(dt), dt, tr)
    np.random.seed(1234)
    u2 = make()
    mask = exact_update_mask(dt, tr.dts)
    pad = lambda col: np.append(col, 0.0)   # noqa: E731
    means, covs, ui = [u2.x.reshape(5, 1).copy()], [np.array(u2.P)], 0
    u2.update(pad(tr.z[:, 0]))
    for s in range(len(dt)):
        u2.predict(dt=dt[s], c=None, sog_rate=tr.sog_rate[ui], cog_rate=tr.cog_rate[ui])
        if mask[s]:
            ui += 1
            u2.update(pad(tr.z[:, ui]))
        means.append(u2.x.reshape(5, 1).copy())
        covs.append(np.array(u2.P))
    assert np.array_equal(m1, np.asarray(means).squeeze()) and np.array_equal(c1, np.asarray(covs).squeeze())
    assert np.array_equal(u1.x, u2.x) and np.array_equal(u1.P, u2.P) and u1.status == u2.status
    after2 = np.random.normal(size=4)
    np.random.seed(1234)
    make().run(len(dt), dt, tr)
    assert np.array_equal(np.random.normal(size=4), after2)   # the same number of draws
    u1.run(len(dt), dt, tr)
    assert len(u1.means) == len(u1.covariances) == 2 * (len(dt) + 1)
