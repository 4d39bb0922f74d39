"""CPU: per-track process noise on the n = 4 passes without a GPU - the new kernels in a warning-free sm_100a compile, the
two additive entry points (prototypes against the header, every refusal before a launch), and the Python layer:
TrackBatch.from_tracks(Q=) / with_noise order, counts, shapes and symmetry, Q through check / copy_from / input_bytes / to,
and the fused pass and the scores refusing a tile with its own Q."""
import ctypes as C
import os
import re
import subprocess
import tempfile
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from _helpers import REPO

HEADER = os.path.join(REPO, "include", "ste_ukf.h")
FAKE = 0x1000


def test_per_track_q_kernels_compile_without_warnings():
    from ship_track_estimators_b200 import build

    flags = [f for f in build.NVCC_FLAGS if f not in ("-shared", "-Xcompiler", "-fPIC")]
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "ste_ukf.cubin")
        proc = subprocess.run([build._nvcc(), *flags, "-cubin", "-Werror", "all-warnings", "-o", out, "ste_ukf.cu"],
                              cwd=build.CSRC, capture_output=True, text=True)
        assert proc.returncode == 0 and "warning" not in proc.stderr.lower(), proc.stderr
        syms = subprocess.run(["cuobjdump", "-symbols", out], capture_output=True, text=True).stdout
    entries = set(re.findall(r"STO_ENTRY\s+(\S+)", syms))
    for pos in "01":
        for gating in "01":
            for innov in "01":
                assert f"_ZN3ste18ukf_forward_kernelILb{pos}ELb{gating}ELb{innov}ELb1EEEvNS_11ForwardArgsIXT1_EXT2_EE4typeE" in entries
    for tape in "01":
        assert f"_ZN3ste21urtss_backward_kernelILb{tape}ELb1EEEvNS_11ForwardArgsILb0EXT0_EE4typeE" in entries
    # the fused kernel and the scores are not instantiated for a per-track Q
    for e in entries:
        if "ukf_roles_kernel" in e or "ukf_score_kernel" in e:
            assert re.search(r"_kernelI(Lb[01]E){2}EEv", e), e


def test_noise_entry_points_match_the_header(native_lib):
    from ship_track_estimators_b200 import _native as nat

    text = open(HEADER).read()
    assert int(re.search(r"#define STE_ABI_VERSION (\d+)", text).group(1)) == nat.STE_ABI_VERSION == native_lib.ste_version() == 7
    expect = {
        "ste_ukf_forward_noise_f64": ["const SteProblem *prob", "const SteInputs *in", "const SteNoiseN *noise",
                                      "const SteInnovations *innov", "SteOutputs *out", "void *stream"],
        "ste_urtss_backward_noise_f64": ["const SteProblem *prob", "const SteInputs *in", "const SteNoiseN *noise", "SteOutputs *out",
                                         "void *stream"],
    }
    ctype = {"SteProblem": nat.SteProblem, "SteInputs": nat.SteInputs, "SteNoiseN": nat.SteNoiseN,
             "SteInnovations": nat.SteInnovations, "SteOutputs": nat.SteOutputs}
    for name, params in expect.items():
        decl = re.search(r"int %s\(([^;]*)\);" % name, text).group(1)
        assert [p.strip() for p in re.sub(r"\s+", " ", decl).split(",")] == params
        restype, argtypes = nat._PROTOTYPES[name]
        assert restype is C.c_int and hasattr(native_lib, name)
        want = [C.c_void_p if p == "void *stream" else C.POINTER(ctype[re.search(r"(Ste\w+)", p).group(1)]) for p in params]
        assert argtypes == want, name


def _tile(nat, n_tracks=0):
    """A valid n = 4 tile with fake device pointers: every check passes, so only the argument under test can refuse (and
    nothing may launch: the tile has no tracks)."""
    p, i, o = nat.SteProblem(), nat.SteInputs(), nat.SteOutputs()
    p.n_tracks, p.max_steps, p.max_obs, p.ld, p.substeps, p.rate_repeat, p.gate_max_iter = n_tracks, 3, 2, 4, 1, 1, 10
    for k in range(4):
        p.H[k * 5] = p.R[k * 5] = 1.0 if k < 2 else 0.0
        p.Q[k * 5] = p.P0[k * 5] = 1.0
    i.x0 = i.dt = i.sog_rate = i.cog_rate = FAKE
    i.z[0] = i.z[1] = FAKE
    o.mean_f, o.cov_f, o.mean_s, o.cov_s, o.status = FAKE, FAKE + 8, FAKE + 16, FAKE + 24, FAKE + 32
    return p, i, o


def test_noise_entry_points_refuse_before_a_launch(native_lib):
    from ship_track_estimators_b200 import _native as nat

    p, i, o = _tile(nat)
    iv = nat.SteInnovations(FAKE, FAKE + 8, FAKE + 16)
    fwd = lambda nz, innov=None: native_lib.ste_ukf_forward_noise_f64(C.byref(p), C.byref(i), nz, innov, C.byref(o), None)  # noqa: E731
    bwd = lambda nz: native_lib.ste_urtss_backward_noise_f64(C.byref(p), C.byref(i), nz, C.byref(o), None)  # noqa: E731
    q_only, r_too, neither = nat.SteNoiseN(FAKE, None), nat.SteNoiseN(FAKE, FAKE), nat.SteNoiseN(None, None)
    for nz in (None, C.byref(neither), C.byref(q_only)):
        assert fwd(nz) == nat.STE_OK
        assert fwd(nz, C.byref(iv)) == nat.STE_OK
        assert bwd(nz) == nat.STE_OK
    # a per-track R in SteNoiseN: at n = 4 it travels in SteInputs.R_tracks
    for nz in (C.byref(r_too), C.byref(nat.SteNoiseN(None, FAKE))):
        assert fwd(nz) == nat.STE_ERR_INVALID_ARG
        assert b"R_tracks" in native_lib.ste_last_error()
        assert bwd(nz) == nat.STE_ERR_INVALID_ARG
        assert b"R_tracks" in native_lib.ste_last_error()
    # the existing checks hold with a per-track Q, for a tile with tracks too (they return before any launch)
    for n_tracks in (0, 4):
        p.n_tracks = n_tracks
        nz = C.byref(q_only)
        assert native_lib.ste_ukf_forward_noise_f64(None, C.byref(i), nz, None, C.byref(o), None) == nat.STE_ERR_INVALID_ARG
        assert native_lib.ste_urtss_backward_noise_f64(C.byref(p), None, nz, C.byref(o), None) == nat.STE_ERR_INVALID_ARG
        holed = nat.SteInnovations(FAKE, None, FAKE + 16)
        assert fwd(nz, C.byref(holed)) == nat.STE_ERR_INVALID_ARG
        assert b"SteInnovations" in native_lib.ste_last_error()
        saved = i.dt
        i.dt = None
        assert fwd(nz) == nat.STE_ERR_INVALID_ARG and bwd(nz) == nat.STE_ERR_INVALID_ARG
        i.dt = saved
        saved = o.mean_s
        o.mean_s = None
        assert bwd(nz) == nat.STE_ERR_INVALID_ARG
        o.mean_s = saved
        p.Q[1] = 0.5   # an asymmetric shared Q
        assert fwd(nz) == nat.STE_ERR_UNSUPPORTED and bwd(nz) == nat.STE_ERR_UNSUPPORTED
        p.Q[1] = 0.0
        p.ld = n_tracks - 1 if n_tracks else -1
        assert fwd(nz) == nat.STE_ERR_INVALID_ARG and bwd(nz) == nat.STE_ERR_INVALID_ARG
        p.ld = 4
        i.R_tracks = FAKE   # a per-track R needs the generic update
        assert fwd(nz) == nat.STE_ERR_INVALID_ARG
        assert b"FORCE_GENERIC" in native_lib.ste_last_error()
        i.R_tracks = None
        p.flags = nat.STE_FLAG_GATING
        i.noise_upd = FAKE
        assert fwd(nz) == nat.STE_ERR_UNSUPPORTED
        i.noise_upd = None
        p.flags = 0
    p.n_tracks = 0


def _tracks(lengths=(6, 3, 5, 8), seed=1):
    rng = np.random.default_rng(seed)
    return [SimpleNamespace(dts=np.ones(m - 1), z=rng.normal(size=(4, m)), sog_rate=np.zeros(m), cog_rate=np.zeros(m))
            for m in lengths]


def _q(i):
    Q = np.diag([1e-2, 2e-2, 1e-3, 4e-3]) * (1.0 + i)
    Q[0, 1] = Q[1, 0] = 5e-3 * (i + 1)
    Q[2, 3] = Q[3, 2] = -1e-4 * (i + 1)
    return Q


def test_from_tracks_q_follows_the_length_sort():
    from ship_track_estimators_b200.batch import TrackBatch

    tr = _tracks()
    qs = [_q(i) for i in range(len(tr))]
    b = TrackBatch.from_tracks(tr, [t.dts for t in tr], device="cpu", Q=qs)
    assert b.order is not None and list(b.order) == [3, 0, 2, 1]
    b.check()
    assert b.Q.shape == (16, 4) and b.Q.dtype == torch.float64
    for j, ship in enumerate(b.order):
        assert np.array_equal(b.Q[:, j].numpy(), qs[ship].reshape(-1))
    unsorted = TrackBatch.from_tracks(tr, [t.dts for t in tr], device="cpu", Q=qs, sort_by_length=False)
    assert np.array_equal(unsorted.Q.numpy(), np.stack([q.reshape(-1) for q in qs], axis=1))
    # both together: R permuted the same way
    rs = [np.diag([1e-3, 1e-3, 0.1, 0.2]) * (1 + i) for i in range(len(tr))]
    both = TrackBatch.from_tracks(tr, [t.dts for t in tr], device="cpu", Q=qs, R=rs)
    for j, ship in enumerate(both.order):
        assert np.array_equal(both.R[:, j].numpy(), rs[ship].reshape(-1))
        assert np.array_equal(both.Q[:, j].numpy(), qs[ship].reshape(-1))


def test_from_tracks_and_with_noise_refuse_bad_matrices():
    from ship_track_estimators_b200.batch import TrackBatch

    tr = _tracks()
    dts = [t.dts for t in tr]
    qs = [_q(i) for i in range(len(tr))]
    asym = _q(0)
    asym[0, 2] = 0.5
    b = TrackBatch.from_tracks(tr, dts, device="cpu")
    for make in (lambda **kw: TrackBatch.from_tracks(tr, dts, device="cpu", **kw), b.with_noise):
        with pytest.raises(ValueError, match="3 matrices for 4 tracks"):
            make(Q=qs[:3])
        with pytest.raises(ValueError, match="5 matrices for 4 tracks"):
            make(Q=qs + [qs[0]])
        with pytest.raises(NotImplementedError, match="shape"):
            make(Q=qs[:3] + [np.eye(5)])
        with pytest.raises(NotImplementedError, match="symmetric"):
            make(Q=qs[:3] + [asym])
    with pytest.raises(ValueError, match="matrices for 4 tracks"):
        b.with_noise(R=qs[:2])
    with pytest.raises(NotImplementedError, match="symmetric"):
        b.with_noise(R=qs[:3] + [asym])


def test_with_noise_places_ship_matrices_by_order_and_shares_the_rest():
    from ship_track_estimators_b200.batch import TrackBatch

    tr = _tracks()
    dts = [t.dts for t in tr]
    qs = [_q(i) for i in range(len(tr))]
    rs = [np.diag([1e-3, 1e-3, 0.1, 0.2]) * (1 + i) for i in range(len(tr))]
    b = TrackBatch.from_tracks(tr, dts, device="cpu")
    assert b.Q is None and b.R is None
    nb = b.with_noise(Q=qs)
    ref = TrackBatch.from_tracks(tr, dts, device="cpu", Q=qs)
    assert torch.equal(nb.Q, ref.Q) and nb.R is None
    for name in ("x0", "dt", "sog_rate", "cog_rate", "upd_mask", "n_steps", "rate_repeat"):
        assert getattr(nb, name) is getattr(b, name)
    assert all(x is y for x, y in zip(nb.z, b.z)) and nb.order is b.order
    assert b.Q is None   # the original tile is unchanged
    both = nb.with_noise(R=rs)   # a set not given keeps the tile's own
    assert both.Q is nb.Q
    assert torch.equal(both.R, TrackBatch.from_tracks(tr, dts, device="cpu", R=rs).R)
    # a tile in the caller's order (no permutation)
    plain = TrackBatch.from_tracks(tr, dts, device="cpu", sort_by_length=False).with_noise(Q=qs)
    assert np.array_equal(plain.Q.numpy(), np.stack([q.reshape(-1) for q in qs], axis=1))


def test_q_travels_with_the_tile():
    from ship_track_estimators_b200.batch import TrackBatch

    tr = _tracks()
    dts = [t.dts for t in tr]
    qs = [_q(i) for i in range(len(tr))]
    b = TrackBatch.from_tracks(tr, dts, device="cpu")
    nb = b.with_noise(Q=qs)
    assert nb.input_bytes() == b.input_bytes() + 16 * 4 * 8
    # check(): shape, dtype, contiguity
    for bad in (nb.Q[:15].clone(), nb.Q.to(torch.float32), nb.Q.t().contiguous().t(), torch.zeros(16, 3, dtype=torch.float64)):
        with pytest.raises(ValueError, match=r"TrackBatch\.Q"):
            TrackBatch(**{**nb.__dict__, "Q": bad}).check()
    # copy_from: the same optional tensors present, or nothing is copied
    dst = TrackBatch.from_tracks(tr, dts, device="cpu", Q=[np.eye(4)] * 4)
    assert dst.copy_from(nb, non_blocking=False)
    assert torch.equal(dst.Q, nb.Q)
    assert not b.copy_from(nb) and not nb.copy_from(b)
    # to(), and with it the host pipeline's staging copies, carries it
    assert torch.equal(nb.to("cpu").Q, nb.Q)


def test_fused_and_score_refuse_a_tile_with_its_own_q(native_lib):
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch

    tr = _tracks()
    dts = [t.dts for t in tr]
    b = TrackBatch.from_tracks(tr, dts, device="cpu")
    nb = b.with_noise(Q=[_q(i) for i in range(len(tr))])
    r4 = np.diag([1e-3, 1e-3, 0.0, 0.0])
    ukf = BatchedUKF(np.diag([1.0, 1.0, 0.0, 0.0]), R=r4)
    with pytest.raises(ValueError, match="per-track process noise"):
        ukf.score(nb, [(np.eye(4), r4)])
    # the refusals come before any buffer is touched: no result sets needed
    with pytest.raises(ValueError, match="per-track Q"):
        ukf.fused(nb, SimpleNamespace(nis=None), b, None)
    with pytest.raises(ValueError, match="per-track Q"):
        ukf.fused(b, SimpleNamespace(nis=None), nb, None)
    with pytest.raises(ValueError, match="per-track Q"):
        ukf.run_many([b, nb], [None, None], fused=True)
