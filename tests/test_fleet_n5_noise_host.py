"""CPU: per-track process and measurement noise on the five-state fleet path without a GPU - the additive C ABI (SteNoiseN
and the two _noise_ entry points, SteInputsN as it was) and its argument checks, the checks of TrackBatchN.from_tracks /
from_batch / check, the matrices following their tracks through the length sort and fleet_tiles, estimate_fleet's ship_settings validation, and a warning-free sm_100a compile."""
import ctypes as C
import os
import re
import subprocess
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest

from _helpers import REPO

HEADER = os.path.join(REPO, "include", "ste_ukf.h")
SETTINGS5 = {"dim": 5, "H": [1, 1, 0, 0, 0], "R": [1e-3] * 5, "Q": [1e-2] * 5, "P": [1.0] * 5, "dt": -1, "nsteps": 1}


def _track(nobs, seed):
    rng = np.random.default_rng(seed)
    return SimpleNamespace(dts=np.ones(nobs - 1), z=rng.normal(size=(4, nobs)), sog_rate=rng.normal(size=nobs), cog_rate=rng.normal(size=nobs))


def _sym(seed):
    """A distinct symmetric 5 x 5 matrix per seed."""
    A = np.random.default_rng(seed).normal(size=(5, 5))
    return A @ A.T + np.eye(5)


def test_noise_entry_points_are_additive(native_lib):
    """The per-track noise travels in its own struct through two new entry points: the version, SteInputsN and the existing
    fleet entry points stay as they were."""
    from ship_track_estimators_b200 import _native as nat

    text = open(HEADER).read()
    assert int(re.search(r"#define STE_ABI_VERSION (\d+)", text).group(1)) == nat.STE_ABI_VERSION == native_lib.ste_version() == 7
    assert [f for f, _ in nat.SteInputsN._fields_][-3:] == ["noise_pred", "noise_upd", "noise_bwd"] and C.sizeof(nat.SteInputsN) == 152
    for name in ("ste_ukf_forward_noise_n_f64", "ste_urtss_backward_tracks_noise_n_f64"):
        decl = re.search(r"int %s\(([^;]*)\);" % name, text).group(1)
        params = [p.strip() for p in decl.split(",")]
        assert params[:3] == ["const SteProblemN *prob", "const SteInputsN *in", "const SteNoiseN *noise"] and len(params) == 5
        restype, argtypes = nat._PROTOTYPES[name]
        assert restype is C.c_int and argtypes[2] == C.POINTER(nat.SteNoiseN) and argtypes[3] == C.POINTER(nat.SteOutputsN)
        assert hasattr(native_lib, name)


def test_noise_entry_points_check_their_arguments_without_a_launch(native_lib):
    """The _noise_ entry points run the fleet path's checks before any launch (here: no GPU, so nothing may launch)."""
    from ship_track_estimators_b200 import _native as nat

    p, i, o, nz = nat.SteProblemN(), nat.SteInputsN(), nat.SteOutputsN(), nat.SteNoiseN(0x1000, 0x2000)
    p.n, p.model, p.n_tracks, p.max_steps, p.max_obs, p.ld = 5, nat.STE_MODEL_GEODETIC_TURN, 4, 3, 2, 4
    for k in range(5):
        p.Q[k * 5 + k] = p.R[k * 5 + k] = p.P0[k * 5 + k] = 1.0
    fwd, bwd = native_lib.ste_ukf_forward_noise_n_f64, native_lib.ste_urtss_backward_tracks_noise_n_f64
    for f in (fwd, bwd):
        assert f(C.byref(p), C.byref(i), C.byref(nz), C.byref(o), None) == nat.STE_ERR_INVALID_ARG   # missing arrays
        assert f(C.byref(p), C.byref(i), None, C.byref(o), None) == nat.STE_ERR_INVALID_ARG
        assert f(None, C.byref(i), C.byref(nz), C.byref(o), None) == nat.STE_ERR_INVALID_ARG
    p.Q[1] = 0.5
    assert fwd(C.byref(p), C.byref(i), C.byref(nz), C.byref(o), None) == nat.STE_ERR_UNSUPPORTED
    assert b"symmetric" in native_lib.ste_last_error()


def test_fleet_structs_match_c_layout():
    """The ctypes mirror of the five-state structs, SteNoiseN included, against the C compiler's offsets."""
    from ship_track_estimators_b200 import _native as nat

    structs = {"SteProblemN": nat.SteProblemN, "SteInputsN": nat.SteInputsN, "SteOutputsN": nat.SteOutputsN, "SteNoiseN": nat.SteNoiseN}
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{HEADER}"', "int main(void){"]
    for sname, cls in structs.items():
        lines.append(f'printf("{sname} %zu\\n", sizeof({sname}));')
        for fname, _ in cls._fields_:
            lines.append(f'printf("{sname}.{fname} %zu\\n", offsetof({sname}, {fname}));')
    lines.append("return 0;}")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "layout.c"), os.path.join(tmp, "layout")
        open(src, "w").write("\n".join(lines))
        subprocess.check_call(["gcc", "-std=c11", src, "-o", exe])
        c_layout = dict(line.split() for line in subprocess.check_output([exe], text=True).strip().splitlines())
    for sname, cls in structs.items():
        assert int(c_layout[sname]) == C.sizeof(cls), sname
        for fname, _ in cls._fields_:
            assert int(c_layout[f"{sname}.{fname}"]) == getattr(cls, fname).offset, f"{sname}.{fname}"
    assert C.sizeof(nat.SteNoiseN) == 16 and nat.SteNoiseN.R_tracks.offset == 8


def test_from_tracks_permutes_and_checks_the_matrices():
    import torch

    from ship_track_estimators_b200.batch_n import TrackBatchN

    lengths = [5, 12, 3, 12, 8]
    tracks = [_track(m, k) for k, m in enumerate(lengths)]
    dts = [t.dts for t in tracks]
    Qs, Rs = [_sym(k) for k in range(5)], [_sym(100 + k) for k in range(5)]
    b = TrackBatchN.from_tracks(tracks, dts, device="cpu", Q=Qs, R=Rs)
    b.check()
    assert b.order is not None and list(b.order) == [1, 3, 4, 0, 2]
    assert b.Q.shape == (25, 5) and b.Q.dtype == torch.float64 and b.Q.is_contiguous()
    for j, i in enumerate(b.order):   # column j holds caller track i, row-major planes
        assert np.array_equal(b.Q[:, j].numpy(), Qs[i].reshape(-1)) and np.array_equal(b.R[:, j].numpy(), Rs[i].reshape(-1))
    unsorted = TrackBatchN.from_tracks(tracks, dts, device="cpu", Q=Qs, sort_by_length=False)
    assert unsorted.R is None and np.array_equal(unsorted.Q.numpy(), np.stack([q.reshape(-1) for q in Qs], axis=1))
    plain = TrackBatchN.from_tracks(tracks, dts, device="cpu")
    assert plain.Q is None and plain.R is None
    assert b.input_bytes() == plain.input_bytes() + 2 * 25 * 8 * len(tracks)   # 400 B per track
    pinned_like = b._map(lambda t: t.clone())
    assert pinned_like.Q is not b.Q and torch.equal(pinned_like.Q, b.Q) and torch.equal(pinned_like.R, b.R)
    assert not plain.copy_from(b)                               # a different layout: nothing copied
    other = TrackBatchN.from_tracks(tracks, dts, device="cpu", Q=Qs[::-1], R=Rs[::-1])
    assert other.copy_from(b, non_blocking=False) and torch.equal(other.Q, b.Q) and torch.equal(other.R, b.R)

    asym = _sym(7)
    asym[0, 4] += 1e-12
    for kw, msg in ((dict(Q=Qs[:4]), "4 matrices for 5 tracks"), (dict(R=Rs + [Rs[0]]), "6 matrices for 5 tracks"),
                    (dict(Q=Qs[:2] + [np.eye(4)] + Qs[3:]), r"Q\[2\] has shape \(4, 4\)"),
                    (dict(R=Rs[:3] + [asym] + Rs[4:]), r"R\[3\] must be symmetric")):
        with pytest.raises(ValueError, match=msg):
            TrackBatchN.from_tracks(tracks, dts, device="cpu", **kw)


def test_check_rejects_a_wrong_plane_count():
    import torch

    from ship_track_estimators_b200.batch_n import TrackBatchN

    tracks = [_track(6, 1), _track(4, 2)]
    b = TrackBatchN.from_tracks(tracks, [t.dts for t in tracks], device="cpu", Q=[np.eye(5)] * 2, R=[np.eye(5)] * 2)
    b.check()
    for name, bad in (("Q", torch.zeros(24, 2, dtype=torch.float64)), ("R", torch.zeros(25, 3, dtype=torch.float64)),
                      ("Q", torch.zeros(25, 2, dtype=torch.float32)), ("R", torch.zeros(2, 25, dtype=torch.float64).T)):
        c = TrackBatchN(**{**b.__dict__, name: bad})
        with pytest.raises(ValueError, match=f"TrackBatchN.{name}"):
            c.check()


def test_from_batch_maps_ship_matrices_through_the_order():
    from ship_track_estimators_b200.batch import TrackBatch
    from ship_track_estimators_b200.batch_n import TrackBatchN

    lengths = [4, 9, 6, 9, 2]
    tracks = [_track(m, 10 + k) for k, m in enumerate(lengths)]
    b4 = TrackBatch.from_tracks(tracks, [t.dts for t in tracks], device="cpu")
    assert b4.order is not None and list(b4.order) != list(range(5))
    Qs, Rs = [_sym(k) for k in range(5)], [_sym(50 + k) for k in range(5)]
    bn = TrackBatchN.from_batch(b4, Q=Qs, R=Rs)
    bn.check()
    for j, i in enumerate(b4.order):
        assert np.array_equal(bn.Q[:, j].numpy(), Qs[i].reshape(-1)) and np.array_equal(bn.R[:, j].numpy(), Rs[i].reshape(-1))
    assert TrackBatchN.from_batch(b4, R=Rs).Q is None
    asym = np.eye(5)
    asym[1, 2] = 0.5
    for kw, msg in ((dict(Q=Qs[:4]), "4 matrices for 5 tracks"), (dict(R=[np.eye(5)] * 4 + [np.eye(6)]), r"R\[4\] has shape"),
                    (dict(Q=[asym] + Qs[1:]), r"Q\[0\] must be symmetric")):
        with pytest.raises(ValueError, match=msg):
            TrackBatchN.from_batch(b4, **kw)
    b4.R = b4.x0.new_zeros(16, 5)   # an n = 4 tile carrying R is still refused, matrices or not
    with pytest.raises(ValueError, match="TrackBatch.R is 4-state data"):
        TrackBatchN.from_batch(b4, Q=Qs)


def test_fleet_tiles_hand_each_tile_its_tracks_matrices():
    from ship_track_estimators_b200.batch_n import TrackBatchN

    rng = np.random.default_rng(9)
    lengths = rng.integers(2, 30, size=41)
    tracks = [_track(int(m), k) for k, m in enumerate(lengths)]
    Qs, Rs = [_sym(k) for k in range(41)], [_sym(500 + k) for k in range(41)]
    tiles = TrackBatchN.fleet_tiles(tracks, [t.dts for t in tracks], device="cpu", state_budget=150, granule=4, Q=Qs, R=Rs)
    assert len(tiles) > 2 and sum(t.n_tracks for t in tiles) == 41
    for tile in tiles:
        tile.check()
        for j, i in enumerate(tile.order):
            assert np.array_equal(tile.Q[:, j].numpy(), Qs[i].reshape(-1)) and np.array_equal(tile.R[:, j].numpy(), Rs[i].reshape(-1))
    with pytest.raises(ValueError, match="matrices for"):
        TrackBatchN.fleet_tiles(tracks, [t.dts for t in tracks], device="cpu", state_budget=150, Q=Qs[:40])


def test_estimate_fleet_ship_settings_are_checked_first(tmp_path):
    """Every ship_settings error is raised before any device work (device="cpu" would fail there): dim 4 and the matrix
    checks before the file is read, an unknown id right after the host parse."""
    from test_host_dropin import _fleet_csv

    from ship_track_estimators_b200.cli import writers

    missing = str(tmp_path / "no_such.csv")
    s4 = {**SETTINGS5, "dim": 4, "H": [1, 1, 0, 0], "R": [1e-3] * 4, "Q": [1e-2] * 4, "P": [1.0] * 4}
    with pytest.raises(NotImplementedError, match=r"TrackBatch.from_tracks\(R=...\).*no per-track Q"):
        writers.estimate_fleet(missing, s4, device="cpu", ship_settings={"1": {"R": [1e-3] * 4}})
    with pytest.raises(FileNotFoundError):   # empty ship_settings: nothing to refuse at dim 4
        writers.estimate_fleet(missing, s4, device="cpu", ship_settings={})
    with pytest.raises(AssertionError, match="Dimension mismatch"):
        writers.estimate_fleet(missing, SETTINGS5, device="cpu", ship_settings={"1": {"Q": [1e-2] * 4}})
    with pytest.raises(AssertionError, match="Dimension mismatch"):
        writers.estimate_fleet(missing, SETTINGS5, device="cpu", ship_settings={"1": {"R": np.eye(5)[:, :4].tolist()}})
    asym = np.eye(5)
    asym[0, 1] = 0.1
    with pytest.raises(ValueError, match="must be symmetric"):
        writers.estimate_fleet(missing, SETTINGS5, device="cpu", ship_settings={"1": {"Q": asym.tolist()}})
    with pytest.raises(ValueError, match="unknown keys"):
        writers.estimate_fleet(missing, SETTINGS5, device="cpu", ship_settings={"1": {"P": [1.0] * 5}})

    csv = str(tmp_path / "fleet.csv")
    _fleet_csv(csv, seed=5, n_ships=6, time_ordered=True)
    from ship_track_estimators_b200.ingest import read_csv_fleet

    ids = read_csv_fleet(csv, id_col="primary.id", on_bad_rows="skip").ids
    with pytest.raises(ValueError, match="not in"):
        writers.estimate_fleet(csv, SETTINGS5, id_col="primary.id", device="cpu",
                               ship_settings={ids[0]: {"R": [0.25] * 5}, "no-such-ship": {"Q": [1e-3] * 5}})


def test_fleet_kernels_compile_without_warnings():
    """ste_ukf.cu for sm_100a with the library's flags and every warning an error; both fleet kernels exist in the shared
    and the per-track form."""
    from ship_track_estimators_b200 import build

    flags = [f for f in build.NVCC_FLAGS if f not in ("-shared", "-Xcompiler", "-fPIC")]
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "ste_ukf.cubin")
        proc = subprocess.run([build._nvcc(), *flags, "-cubin", "-Werror", "all-warnings", "-o", out, "ste_ukf.cu"],
                              cwd=build.CSRC, capture_output=True, text=True)
        assert proc.returncode == 0 and "warning" not in proc.stderr.lower(), proc.stderr
        syms = subprocess.run(["cuobjdump", "-symbols", out], capture_output=True, text=True).stdout
    for kernel in ("ukf_forward_n_kernelILi5ELb0E", "ukf_forward_n_kernelILi5ELb1E", "urtss_backward_n_tracks_kernelILi5ELb0E",
                   "urtss_backward_n_tracks_kernelILi5ELb1E"):
        assert kernel in syms, kernel
