"""CPU: the innovation statistics without a GPU - the additive C ABI (SteInnovations and the two _innov_ entry points,
every existing struct as it was) and its argument checks, the new kernel instantiations in a warning-free sm_100a compile,
allocate(innovations=True), the shape checks, innovation_metrics' masking and the fused pass refusing the planes."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from _helpers import REPO

HEADER = os.path.join(REPO, "include", "ste_ukf.h")


def test_innovation_entry_points_are_additive(native_lib):
    from ship_track_estimators_b200 import _native as nat

    text = open(HEADER).read()
    assert int(re.search(r"#define STE_ABI_VERSION (\d+)", text).group(1)) == nat.STE_ABI_VERSION == native_lib.ste_version() == 7
    sizes = {nat.SteProblem: 560, nat.SteInputs: 128, nat.SteOutputs: 80, nat.SteProblemN: 2080, nat.SteInputsN: 152,
             nat.SteOutputsN: 48, nat.SteNoiseN: 16, nat.SteInnovations: 24}
    for cls, size in sizes.items():
        assert C.sizeof(cls) == size, cls.__name__
    decls = {"ste_ukf_forward_innov_f64": ["const SteProblem *prob", "const SteInputs *in", "const SteInnovations *innov",
                                           "SteOutputs *out", "void *stream"],
             "ste_ukf_forward_innov_n_f64": ["const SteProblemN *prob", "const SteInputsN *in", "const SteNoiseN *noise",
                                             "const SteInnovations *innov", "SteOutputsN *out", "void *stream"]}
    for name, params in decls.items():
        decl = re.search(r"int %s\(([^;]*)\);" % name, text).group(1)
        assert [p.strip() for p in decl.split(",")] == params
        restype, argtypes = nat._PROTOTYPES[name]
        assert restype is C.c_int and C.POINTER(nat.SteInnovations) in argtypes and hasattr(native_lib, name)


def test_innovations_struct_matches_c_layout():
    from ship_track_estimators_b200 import _native as nat

    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{HEADER}"', "int main(void){",
             'printf("size %zu\\n", sizeof(SteInnovations));']
    lines += [f'printf("{f} %zu\\n", offsetof(SteInnovations, {f}));' for f, _ in nat.SteInnovations._fields_]
    lines.append("return 0;}")
    with tempfile.TemporaryDirectory() as tmp:
        src, exe = os.path.join(tmp, "layout.c"), os.path.join(tmp, "layout")
        open(src, "w").write("\n".join(lines))
        subprocess.check_call(["gcc", "-std=c11", src, "-o", exe])
        layout = dict(line.split() for line in subprocess.check_output([exe], text=True).strip().splitlines())
    assert int(layout["size"]) == C.sizeof(nat.SteInnovations)
    for f, _ in nat.SteInnovations._fields_:
        assert int(layout[f]) == getattr(nat.SteInnovations, f).offset, f


def test_innovation_entry_points_check_their_arguments_without_a_launch(native_lib):
    """Every check runs before any launch (no GPU here: nothing may launch)."""
    from ship_track_estimators_b200 import _native as nat

    fake = 0x1000
    p4, i4, o4 = nat.SteProblem(), nat.SteInputs(), nat.SteOutputs()
    p4.n_tracks, p4.max_steps, p4.max_obs, p4.ld, p4.substeps, p4.rate_repeat = 4, 3, 2, 4, 1, 1
    for k in range(4):
        p4.H[k * 5] = p4.R[k * 5] = 1.0 if k < 2 else 0.0   # the position-only update: rows 0 and 1 only
        p4.Q[k * 5] = p4.P0[k * 5] = 1.0
    pn, i_n, on = nat.SteProblemN(), nat.SteInputsN(), nat.SteOutputsN()
    pn.n, pn.model, pn.n_tracks, pn.max_steps, pn.max_obs, pn.ld = 5, nat.STE_MODEL_GEODETIC_TURN, 4, 3, 2, 4
    for k in range(5):
        pn.Q[k * 5 + k] = pn.R[k * 5 + k] = pn.P0[k * 5 + k] = 1.0
    full, holed = nat.SteInnovations(fake, fake, fake), nat.SteInnovations(fake, None, fake)
    f4 = lambda p, i, v, o: native_lib.ste_ukf_forward_innov_f64(p, i, v, o, None)   # noqa: E731
    f5 = lambda p, i, v, o: native_lib.ste_ukf_forward_innov_n_f64(p, i, None, v, o, None)   # noqa: E731
    for f, p, i, o in ((f4, p4, i4, o4), (f5, pn, i_n, on)):
        assert f(None, C.byref(i), C.byref(full), C.byref(o)) == nat.STE_ERR_INVALID_ARG
        assert f(C.byref(p), C.byref(i), C.byref(full), C.byref(o)) == nat.STE_ERR_INVALID_ARG   # missing arrays
        assert f(C.byref(p), C.byref(i), None, C.byref(o)) == nat.STE_ERR_INVALID_ARG
    # every array present: a plane missing from innov is the only error left
    i4.x0 = i4.dt = i4.sog_rate = i4.cog_rate = fake
    i4.z[0] = i4.z[1] = fake
    o4.mean_f = o4.cov_f = o4.status = fake
    i_n.x0 = i_n.dt = i_n.sog_rate = i_n.upd_mask = fake
    on.mean_f, on.cov_f, on.status = fake, fake + 8, fake + 16
    for f, p, i, o in ((f4, p4, i4, o4), (f5, pn, i_n, on)):
        for v in (holed, nat.SteInnovations(None, fake, fake), nat.SteInnovations(fake, fake, None)):
            assert f(C.byref(p), C.byref(i), C.byref(v), C.byref(o)) == nat.STE_ERR_INVALID_ARG
            assert b"SteInnovations" in native_lib.ste_last_error()
        p.Q[1] = 0.5   # an asymmetric Q is still refused as unsupported
        assert f(C.byref(p), C.byref(i), C.byref(full), C.byref(o)) == nat.STE_ERR_UNSUPPORTED
        assert b"symmetric" in native_lib.ste_last_error()


def test_innovation_kernels_compile_without_warnings():
    """ste_ukf.cu for sm_100a with the library's flags and every warning an error; both forward kernels exist in their
    statistics-writing form beside the existing ones."""
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
            for innov in "01":
                assert f"ukf_forward_kernelILb{pos}ELb{gating}ELb{innov}E" in syms
    for per_track in "01":
        for innov in "01":
            assert f"ukf_forward_n_kernelILi5ELb{per_track}ELb{innov}E" in syms


def _tile4():
    from types import SimpleNamespace

    from ship_track_estimators_b200.batch import TrackBatch

    rng = np.random.default_rng(1)
    tracks = [SimpleNamespace(dts=np.ones(m - 1), z=rng.normal(size=(4, m)), sog_rate=np.zeros(m), cog_rate=np.zeros(m))
              for m in (6, 3, 5)]
    return TrackBatch.from_tracks(tracks, [t.dts for t in tracks], device="cpu"), tracks


def test_allocate_innovations_and_the_shape_checks(native_lib):
    import torch

    from ship_track_estimators_b200.batch import BatchedUKF, TrackResults
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN

    b, tracks = _tile4()
    ukf = BatchedUKF(np.diag([1.0, 1.0, 0.0, 0.0]), R=np.diag([1e-3, 1e-3, 0.0, 0.0]))
    plain, res = ukf.allocate(b), ukf.allocate(b, innovations=True)
    assert plain.nis is None and plain.loglik is None and plain.innov_rank is None
    for name, dtype in (("nis", torch.float64), ("loglik", torch.float64), ("innov_rank", torch.uint8)):
        t = getattr(res, name)
        assert t.shape == (b.max_obs, b.n_tracks) and t.dtype == dtype and t.is_contiguous()
    ukf._check_shapes(b, res)
    host = res.host_like(pinned=False)
    assert host.nis.shape == res.nis.shape and host.innov_rank.dtype == torch.uint8
    assert res.copy_to(host, non_blocking=False) > 0 and torch.equal(host.innov_rank, res.innov_rank)
    for name, bad in (("nis", torch.zeros(b.max_obs + 1, b.n_tracks, dtype=torch.float64)),
                      ("loglik", torch.zeros(b.max_obs, b.n_tracks, dtype=torch.float32)),
                      ("innov_rank", torch.zeros(b.max_obs, b.n_tracks, dtype=torch.int32)),
                      ("nis", torch.zeros(b.n_tracks, b.max_obs, dtype=torch.float64).T)):
        broken = TrackResults(**{**res.__dict__, name: bad})
        with pytest.raises(ValueError, match=f"TrackResults.{name}"):
            ukf._check_shapes(b, broken)
    with pytest.raises(ValueError, match="allocated together"):
        ukf._check_shapes(b, TrackResults(**{**res.__dict__, "loglik": None}))

    tracks5 = [type(t)(dts=t.dts, z=np.vstack([t.z, np.zeros((1, t.z.shape[1]))]), sog_rate=t.sog_rate, cog_rate=t.cog_rate)
               for t in tracks]
    b5 = TrackBatchN.from_tracks(tracks5, [t.dts for t in tracks5], device="cpu")
    engine = BatchedUKFN(np.diag([1.0, 1.0, 0.0, 0.0, 0.0]))
    r5 = engine.allocate(b5, innovations=True)
    assert r5.nis.shape == (b5.max_obs, b5.n_tracks) and r5.innov_rank.dtype == torch.uint8
    engine._check_shapes(b5, r5)
    assert engine.allocate(b5).nis is None
    with pytest.raises(ValueError, match="TrackResultsN.innov_rank"):
        engine._check_shapes(b5, type(r5)(**{**r5.__dict__, "innov_rank": r5.nis}))


def test_track_keys_and_innovation_metrics_masking(native_lib):
    """innovation_metrics sums only rows below each track's n_updates (garbage beyond them) and keeps column order."""
    import torch

    from ship_track_estimators_b200.batch import BatchedUKF
    from ship_track_estimators_b200.performance_metrics import innovation_metrics

    b, _ = _tile4()
    ukf = BatchedUKF(np.diag([1.0, 1.0, 0.0, 0.0]))
    res = ukf.allocate(b, innovations=True, smoother=False)
    M, T = res.nis.shape
    res.n_updates.copy_(torch.tensor([M, 2, 0], dtype=torch.int32))
    res.mean_f.zero_()
    res.cov_f.zero_()
    res.nis.copy_(torch.arange(M * T, dtype=torch.float64).reshape(M, T))
    res.loglik.copy_(-res.nis)
    res.innov_rank.fill_(2)
    for t in range(T):   # garbage where no update wrote
        res.nis[int(res.n_updates[t]):, t] = float("inf")
        res.loglik[int(res.n_updates[t]):, t] = float("nan")
        res.innov_rank[int(res.n_updates[t]):, t] = 255
    m = innovation_metrics(res)
    nis = res.nis.numpy()
    want = [sum(nis[u, t] for u in range(int(res.n_updates[t]))) for t in range(T)]
    assert np.array_equal(m["nis"].numpy(), np.array(want)) and np.array_equal(m["loglik"].numpy(), -np.array(want))
    assert m["dof"].tolist() == [2 * M, 4, 0] and m["n_updates"].tolist() == [M, 2, 0]
    assert all(v.shape == (T,) for v in m.values())
    got = res.track(b.order[1] if b.order is not None else 1)
    assert np.array_equal(got["nis"], nis[:2, 1]) and got["innov_rank"].tolist() == [2, 2]
    plain = ukf.allocate(b, smoother=False)
    plain.n_updates.fill_(1)
    assert "nis" not in plain.track(0) and "loglik" not in plain.track(0)
    with pytest.raises(ValueError, match="no innovation statistics"):
        innovation_metrics(plain)


def test_fused_pass_refuses_innovation_planes(native_lib):
    from ship_track_estimators_b200.batch import BatchedUKF

    b, _ = _tile4()
    ukf = BatchedUKF(np.diag([1.0, 1.0, 0.0, 0.0]))
    with pytest.raises(ValueError, match="innovation"):
        ukf.fused(b, ukf.allocate(b, innovations=True), b, ukf.allocate(b))
