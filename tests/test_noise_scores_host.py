"""CPU: noise-candidate scores without a GPU - the scoring kernels in a warning-free sm_100a compile, the additive C ABI
(SteCandidates / SteScores against gcc's layout, the two score entry points) and every refusal before a launch, the
Python checks of BatchedUKF.score / BatchedUKFN.score, noise_grid's order and the maximum-likelihood selection rules."""
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


def test_score_kernels_compile_without_warnings():
    from ship_track_estimators_b200 import build

    flags = [f for f in build.NVCC_FLAGS if f not in ("-shared", "-Xcompiler", "-fPIC")]
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "ste_ukf.cubin")
        proc = subprocess.run([build._nvcc(), *flags, "-cubin", "-Werror", "all-warnings", "-o", out, "ste_ukf.cu"],
                              cwd=build.CSRC, capture_output=True, text=True)
        assert proc.returncode == 0 and "warning" not in proc.stderr.lower(), proc.stderr
        syms = subprocess.run(["cuobjdump", "-symbols", out], capture_output=True, text=True).stdout
    for pos in "01":
        for gating in "01":
            assert f"ukf_score_kernelILb{pos}ELb{gating}EE" in syms
    assert "ukf_score_n_kernelILi5EE" in syms


def test_score_abi_is_additive(native_lib):
    from ship_track_estimators_b200 import _native as nat

    text = open(HEADER).read()
    assert int(re.search(r"#define STE_ABI_VERSION (\d+)", text).group(1)) == nat.STE_ABI_VERSION == native_lib.ste_version() == 7
    assert int(re.search(r"#define STE_MAX_CANDIDATES (\d+)", text).group(1)) == nat.STE_MAX_CANDIDATES == 32
    sizes = {nat.SteProblem: 560, nat.SteInputs: 128, nat.SteOutputs: 80, nat.SteProblemN: 2080, nat.SteInputsN: 152,
             nat.SteOutputsN: 48, nat.SteNoiseN: 16, nat.SteInnovations: 24, nat.SteCandidates: 24, nat.SteScores: 48}
    for cls, size in sizes.items():
        assert C.sizeof(cls) == size, cls.__name__
    for name, prob, inputs in (("ste_ukf_score_f64", "SteProblem", "SteInputs"), ("ste_ukf_score_n_f64", "SteProblemN", "SteInputsN")):
        decl = re.search(r"int %s\(([^;]*)\);" % name, text).group(1)
        assert [p.strip() for p in decl.split(",")] == [f"const {prob} *prob", f"const {inputs} *in", "const SteCandidates *cand",
                                                        "SteScores *scores", "void *stream"]
        restype, argtypes = nat._PROTOTYPES[name]
        assert restype is C.c_int and C.POINTER(nat.SteCandidates) in argtypes and hasattr(native_lib, name)


def test_score_structs_match_c_layout():
    from ship_track_estimators_b200 import _native as nat

    structs = {"SteCandidates": nat.SteCandidates, "SteScores": nat.SteScores}
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{HEADER}"', "int main(void){"]
    for sname, cls in structs.items():
        lines.append(f'printf("{sname} %zu\\n", sizeof({sname}));')
        lines += [f'printf("{sname}.{f} %zu\\n", offsetof({sname}, {f}));' for f, _ in cls._fields_]
    lines.append("return 0;}")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "layout.c"), os.path.join(tmp, "layout")
        open(src, "w").write("\n".join(lines))
        subprocess.check_call(["gcc", "-std=c11", src, "-o", exe])
        layout = dict(line.split() for line in subprocess.check_output([exe], text=True).strip().splitlines())
    for sname, cls in structs.items():
        assert int(layout[sname]) == C.sizeof(cls), sname
        for f, _ in cls._fields_:
            assert int(layout[f"{sname}.{f}"]) == getattr(cls, f).offset, f"{sname}.{f}"


FAKE = 0x1000


def _tile_args(nat):
    """A valid n = 4 and n = 5 problem with fake device pointers: every check passes, so nothing but the argument under
    test can refuse (and nothing may launch here: the tiles have no tracks)."""
    p4, i4 = nat.SteProblem(), nat.SteInputs()
    p4.n_tracks, p4.max_steps, p4.max_obs, p4.ld, p4.substeps, p4.rate_repeat, p4.gate_max_iter = 0, 3, 2, 4, 1, 1, 10
    for k in range(4):
        p4.H[k * 5] = p4.R[k * 5] = 1.0 if k < 2 else 0.0
        p4.Q[k * 5] = p4.P0[k * 5] = 1.0
    i4.x0 = i4.dt = i4.sog_rate = i4.cog_rate = FAKE
    i4.z[0] = i4.z[1] = FAKE
    pn, i_n = nat.SteProblemN(), nat.SteInputsN()
    pn.n, pn.model, pn.n_tracks, pn.max_steps, pn.max_obs, pn.ld = 5, nat.STE_MODEL_GEODETIC_TURN, 0, 3, 2, 4
    for k in range(5):
        pn.Q[k * 5 + k] = pn.R[k * 5 + k] = pn.P0[k * 5 + k] = 1.0
    i_n.x0 = i_n.dt = i_n.sog_rate = i_n.upd_mask = FAKE
    return (p4, i4), (pn, i_n)


def _table(nat, mats_q, mats_r, n_cand=None):
    Q = np.ascontiguousarray(np.stack([np.asarray(m, dtype=np.float64).reshape(-1) for m in mats_q]))
    R = np.ascontiguousarray(np.stack([np.asarray(m, dtype=np.float64).reshape(-1) for m in mats_r]))
    dp = C.POINTER(C.c_double)
    cand = nat.SteCandidates(len(Q) if n_cand is None else n_cand, 0, Q.ctypes.data_as(dp), R.ctypes.data_as(dp))
    cand._keep = (Q, R)
    return cand


def test_score_refusals_without_a_launch(native_lib):
    from ship_track_estimators_b200 import _native as nat

    (p4, i4), (pn, i_n) = _tile_args(nat)
    q4, r4 = np.diag([1.0, 1.0, 1e-2, 1e-2]), np.diag([1e-3, 1e-3, 0.0, 0.0])
    q5, r5 = np.eye(5), np.diag([1e-3, 1e-3, 0.0, 0.0, 0.0])
    sc = nat.SteScores(FAKE, FAKE + 8, FAKE + 16, FAKE + 24, FAKE + 32, 4)
    f4 = lambda p, i, cand, s: native_lib.ste_ukf_score_f64(p, i, cand, s, None)    # noqa: E731
    f5 = lambda p, i, cand, s: native_lib.ste_ukf_score_n_f64(p, i, cand, s, None)  # noqa: E731
    for f, p, i, q, r in ((f4, p4, i4, q4, r4), (f5, pn, i_n, q5, r5)):
        good = _table(nat, [q] * 3, [r] * 3)
        assert f(C.byref(p), C.byref(i), C.byref(good), C.byref(sc)) == nat.STE_OK
        # the candidate count
        for n in (0, -1, 33):
            assert f(C.byref(p), C.byref(i), C.byref(_table(nat, [q] * 33, [r] * 33, n_cand=n)), C.byref(sc)) == nat.STE_ERR_INVALID_ARG
        assert f(C.byref(p), C.byref(i), C.byref(_table(nat, [q] * 32, [r] * 32)), C.byref(sc)) == nat.STE_OK
        # NULL table, matrices, outputs; ld_out
        assert f(C.byref(p), C.byref(i), None, C.byref(sc)) == nat.STE_ERR_INVALID_ARG
        for field in ("Q", "R"):
            holed = _table(nat, [q], [r])
            setattr(holed, field, None)
            assert f(C.byref(p), C.byref(i), C.byref(holed), C.byref(sc)) == nat.STE_ERR_INVALID_ARG
        assert f(C.byref(p), C.byref(i), C.byref(good), None) == nat.STE_ERR_INVALID_ARG
        for field in ("loglik", "nis", "dof", "n_updates", "status"):
            holed = nat.SteScores(FAKE, FAKE + 8, FAKE + 16, FAKE + 24, FAKE + 32, 4)
            setattr(holed, field, None)
            assert f(C.byref(p), C.byref(i), C.byref(good), C.byref(holed)) == nat.STE_ERR_INVALID_ARG
            assert b"SteScores" in native_lib.ste_last_error()
        p.n_tracks = 4
        short = nat.SteScores(FAKE, FAKE + 8, FAKE + 16, FAKE + 24, FAKE + 32, 3)
        assert f(C.byref(p), C.byref(i), C.byref(good), C.byref(short)) == nat.STE_ERR_INVALID_ARG
        p.n_tracks = 0
        # asymmetric or non-finite candidates
        bad_q = q.copy()
        bad_q[0, 1] = 0.5
        assert f(C.byref(p), C.byref(i), C.byref(_table(nat, [q, bad_q], [r, r])), C.byref(sc)) == nat.STE_ERR_UNSUPPORTED
        assert b"symmetric" in native_lib.ste_last_error()
        for bad in (np.nan, np.inf):
            bad_r = r.copy()
            bad_r[1, 1] = bad
            assert f(C.byref(p), C.byref(i), C.byref(_table(nat, [q, q], [r, bad_r])), C.byref(sc)) == nat.STE_ERR_UNSUPPORTED
        # a missing input array
        saved = i.dt
        i.dt = None
        assert f(C.byref(p), C.byref(i), C.byref(good), C.byref(sc)) == nat.STE_ERR_INVALID_ARG
        i.dt = saved
    # n = 4: candidates selecting different updates
    generic_r = np.diag([1e-3, 1e-3, 0.5, 4.0])
    i4.z[2] = i4.z[3] = FAKE
    mixed = _table(nat, [q4, q4], [r4, generic_r])
    assert f4(C.byref(p4), C.byref(i4), C.byref(mixed), C.byref(sc)) == nat.STE_ERR_UNSUPPORTED
    assert f4(C.byref(p4), C.byref(i4), C.byref(_table(nat, [q4, q4], [generic_r, generic_r])), C.byref(sc)) == nat.STE_OK
    p4.flags = nat.STE_FLAG_FORCE_GENERIC   # every candidate generic: no split needed
    assert f4(C.byref(p4), C.byref(i4), C.byref(mixed), C.byref(sc)) == nat.STE_OK
    # a row a generic candidate reads is absent
    i4.z[3] = None
    assert f4(C.byref(p4), C.byref(i4), C.byref(_table(nat, [q4], [generic_r])), C.byref(sc)) == nat.STE_ERR_INVALID_ARG
    i4.z[3] = FAKE
    # a tile carrying its own R
    i4.R_tracks = FAKE
    assert f4(C.byref(p4), C.byref(i4), C.byref(_table(nat, [q4], [generic_r])), C.byref(sc)) == nat.STE_ERR_INVALID_ARG
    assert b"R_tracks" in native_lib.ste_last_error()
    i4.R_tracks = None
    # gating with measurement noise tapes, as the forward pass refuses it
    p4.flags = nat.STE_FLAG_GATING
    i4.noise_upd = FAKE
    assert f4(C.byref(p4), C.byref(i4), C.byref(_table(nat, [q4], [r4])), C.byref(sc)) == nat.STE_ERR_UNSUPPORTED
    i4.noise_upd = None
    assert f4(C.byref(p4), C.byref(i4), C.byref(_table(nat, [q4], [r4])), C.byref(sc)) == nat.STE_OK


def _tracks(n_rows, lengths=(6, 3, 5), seed=1):
    rng = np.random.default_rng(seed)
    return [SimpleNamespace(dts=np.ones(m - 1), z=rng.normal(size=(n_rows, m)), sog_rate=np.zeros(m), cog_rate=np.zeros(m))
            for m in lengths]


def test_python_score_checks(native_lib):
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    tr4 = _tracks(4)
    b = TrackBatch.from_tracks(tr4, [t.dts for t in tr4], device="cpu")
    ukf = BatchedUKF(np.diag([1.0, 1.0, 0.0, 0.0]), R=np.diag([1e-3, 1e-3, 0.0, 0.0]))
    q4, r4 = np.eye(4), np.diag([1e-3, 1e-3, 0.0, 0.0])
    with pytest.raises(ValueError, match="no noise candidates"):
        ukf.score(b, [])
    with pytest.raises(ValueError, match="pair"):
        ukf.score(b, [(q4, r4, q4)])
    with pytest.raises(NotImplementedError, match="shape"):
        ukf.score(b, [(np.eye(5), r4)])
    asym = q4.copy()
    asym[0, 1] = 0.1
    with pytest.raises(NotImplementedError, match="symmetric"):
        ukf.score(b, [(q4, r4), (asym, r4)])
    with pytest.raises(ValueError, match="finite"):
        ukf.score(b, [(q4 + np.diag([np.inf, 0.0, 0.0, 0.0]), r4)])   # NaN would fail the symmetry check first
    holed = TrackBatch(**{**b.__dict__, "z": [b.z[0], b.z[1], None, None]})
    with pytest.raises(ValueError, match="row 2"):
        ukf.score(holed, [(q4, np.diag([1e-3, 1e-3, 0.5, 0.0]))])
    with pytest.raises(ValueError, match="per-track"):
        ukf.score(TrackBatch.from_tracks(tr4, [t.dts for t in tr4], device="cpu", R=[r4 + np.diag([0, 0, 1.0, 1.0])] * 3), [(q4, r4)])
    gated = BatchedUKF(np.diag([1.0, 1.0, 0.0, 0.0]), R=r4, gating=True)
    noisy = TrackBatch.from_tracks(tr4, [t.dts for t in tr4], device="cpu", noise=[dict(upd=np.zeros((t.z.shape[1], 4))) for t in tr4])
    with pytest.raises(NotImplementedError, match="gating"):
        gated.score(noisy, [(q4, r4)])

    tr5 = _tracks(5)
    b5 = TrackBatchN.from_tracks(tr5, [t.dts for t in tr5], device="cpu")
    engine = BatchedUKFN(np.diag([1.0, 1.0, 0.0, 0.0, 0.0]))
    q5, r5 = np.eye(5), np.diag([1e-3, 1e-3, 0.0, 0.0, 0.0])
    with pytest.raises(ValueError, match="5 x 5"):
        engine.score(b5, [(q4, r4)])
    asym5 = q5.copy()
    asym5[4, 0] = 0.1
    with pytest.raises(ValueError, match="symmetric"):
        engine.score(b5, [(asym5, r5)])
    with pytest.raises(ValueError, match="finite"):
        engine.score(b5, [(q5, r5 + np.diag([0.0, np.inf, 0.0, 0.0, 0.0]))])
    with pytest.raises(ValueError, match="per-track"):
        engine.score(TrackBatchN.from_tracks(tr5, [t.dts for t in tr5], device="cpu", R=[r5] * 3), [(q5, r5)])
    with pytest.raises(ValueError, match="per-track"):
        engine.score(TrackBatchN.from_tracks(tr5, [t.dts for t in tr5], device="cpu", Q=[q5] * 3), [(q5, r5)])


def test_noise_grid_is_q_major():
    from ship_track_estimators_b200.tuning import noise_grid

    Q, R = np.diag([1.0, 2.0]), np.diag([3.0, 5.0])
    grid = noise_grid(Q, R, (1, 10), (0.5, 2, 4))
    assert len(grid) == 6
    for i, q in enumerate((1, 10)):
        for j, r in enumerate((0.5, 2, 4)):
            gq, gr = grid[i * 3 + j]
            assert np.array_equal(gq, q * Q) and np.array_equal(gr, r * R) and gq.dtype == np.float64


def test_selection_rules():
    from ship_track_estimators_b200.tuning import select_noise

    nan, inf = float("nan"), float("inf")
    L = np.array([[-1.0, -5.0, nan, -2.0],
                  [-3.0, -1.0, -1.0, -2.0],
                  [-1.0, -4.0, -9.0, -inf]])
    fleet = select_noise(L, "fleet")
    # tracks 2 (NaN under candidate 0) and 3 (-inf under candidate 2) are excluded from every sum
    assert fleet["excluded"].tolist() == [2, 3]
    assert np.array_equal(fleet["loglik"], np.array([-6.0, -4.0, -5.0])) and fleet["best"] == 1
    track = select_noise(L, "track")
    # track 0: a tie between 0 and 2 goes to 0; track 2: NaN counts as -inf; track 3: a tie between 0 and 1
    assert track["best"].tolist() == [0, 1, 1, 0] and track["excluded"].tolist() == [2, 3]
    assert track["loglik"] is not None and track["loglik"].shape == (3, 4)
    # a fleet tie goes to the lowest index
    assert select_noise(np.array([[-1.0, -1.0], [-2.0, 0.0]]), "fleet")["best"] == 0
    with pytest.raises(ValueError, match="no track"):
        select_noise(np.array([[nan], [-1.0]]), "fleet")
    assert select_noise(np.array([[nan], [-1.0]]), "track")["best"].tolist() == [1]
    with pytest.raises(ValueError, match="per"):
        select_noise(L, "ship")


class _FakeEngine:
    """score() from a table indexed by caller track: what fit_noise sees from the device, here without one."""

    def __init__(self, table):
        self.table = table

    def score(self, tile, candidates):
        import torch

        assert len(candidates) == self.table.shape[0]
        cols = np.asarray(tile.order)
        return {"loglik": torch.from_numpy(self.table[:, cols].copy())}


def test_fit_noise_maps_tiles_to_caller_order():
    from ship_track_estimators_b200.tuning import fit_noise

    rng = np.random.default_rng(5)
    table = rng.normal(size=(4, 9))
    table[2, 7] = np.nan
    cands = [(np.eye(5) * k, np.eye(5) * (k + 1)) for k in range(4)]
    tiles = [SimpleNamespace(n_tracks=4, order=np.array([8, 3, 0, 5])), SimpleNamespace(n_tracks=5, order=np.array([1, 7, 2, 6, 4]))]
    eng = _FakeEngine(table)
    per_track = fit_noise(eng, tiles, cands, per="track")
    want = np.argmax(np.where(np.isfinite(table), table, -np.inf), axis=0)
    assert per_track["best"].tolist() == want.tolist()
    assert np.array_equal(per_track["loglik"], table, equal_nan=True) and per_track["excluded"].tolist() == [7]
    assert all(np.array_equal(per_track["Q"][i], cands[k][0]) and np.array_equal(per_track["R"][i], cands[k][1]) for i, k in enumerate(want))
    fleet = fit_noise(eng, tiles, cands, per="fleet")
    keep = np.arange(9) != 7
    assert np.array_equal(fleet["loglik"], table[:, keep].sum(axis=1)) and fleet["best"] == int(np.argmax(table[:, keep].sum(axis=1)))
    assert fleet["Q"] is cands[fleet["best"]][0] and fleet["excluded"].tolist() == [7]
    with pytest.raises(ValueError, match="exactly once"):
        fit_noise(eng, [tiles[0], SimpleNamespace(n_tracks=5, order=np.array([1, 7, 2, 6, 6]))], cands)
