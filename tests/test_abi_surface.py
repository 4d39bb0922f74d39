"""CPU: the C-ABI shared library builds for sm_100a, loads without a GPU, exports every symbol
declared in include/ste_ukf.h, and the ctypes mirror of its structs matches the C layout.
No compute calls here (no GPU); invalid-argument paths that return before any launch are checked."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import pytest

from _helpers import REPO

HEADER = os.path.join(REPO, "include", "ste_ukf.h")


def _declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ste_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(native_lib):
    names = _declared_functions()
    assert {"ste_ukf_forward_f64", "ste_urtss_backward_f64", "ste_ukf_predict_f64", "ste_ukf_update_f64",
            "ste_sigma_points_f64", "ste_geodetic_f64", "ste_version", "ste_last_error"} <= set(names)
    for n in names:
        assert hasattr(native_lib, n), f"libste_ukf.so does not export {n}"
    from ship_track_estimators_b200 import _native

    assert set(_native._PROTOTYPES) == set(names), "ctypes prototypes out of sync with the header"
    assert native_lib.ste_version() == _native.STE_ABI_VERSION


def test_library_is_sm100a_only(native_lib):
    from ship_track_estimators_b200 import build

    out = subprocess.run(["cuobjdump", "--list-elf", build.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs


def test_staleness_check_watches_every_included_file():
    """build.is_stale() must see an edit to any file the compile reads: every local #include reachable from the sources."""
    from ship_track_estimators_b200 import build

    todo = [os.path.join(build.CSRC, s) for s in build.SOURCES]
    seen = set()
    while todo:
        path = os.path.normpath(todo.pop())
        if path in seen:
            continue
        seen.add(path)
        for inc in re.findall(r'^\s*#\s*include\s+"([^"]+)"', open(path).read(), flags=re.M):
            todo.append(os.path.join(os.path.dirname(path), inc))
    watched = {os.path.normpath(os.path.join(build.CSRC, f)) for f in build.SOURCES + build.HEADERS}
    assert seen <= watched, sorted(seen - watched)


def test_ctypes_structs_match_c_layout():
    from ship_track_estimators_b200 import _native as nat

    structs = {"SteProblem": nat.SteProblem, "SteInputs": nat.SteInputs, "SteOutputs": nat.SteOutputs}
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


def test_invalid_arguments_return_codes_without_gpu(native_lib):
    from ship_track_estimators_b200 import _native as nat

    p, i, o = nat.SteProblem(), nat.SteInputs(), nat.SteOutputs()
    p.n_tracks, p.max_steps, p.max_obs, p.ld = 4, 2, 0, 4
    assert native_lib.ste_ukf_forward_f64(C.byref(p), C.byref(i), C.byref(o), None) == nat.STE_ERR_INVALID_ARG
    p.max_obs, p.ld = 3, 2  # ld < n_tracks
    assert native_lib.ste_ukf_forward_f64(C.byref(p), C.byref(i), C.byref(o), None) == nat.STE_ERR_INVALID_ARG
    p.ld = 4
    p.Q[1] = 0.5  # asymmetric Q
    assert native_lib.ste_urtss_backward_f64(C.byref(p), C.byref(i), C.byref(o), None) == nat.STE_ERR_UNSUPPORTED
    assert b"symmetric" in native_lib.ste_last_error()
    p.Q[1] = 0.0
    assert native_lib.ste_ukf_forward_f64(C.byref(p), C.byref(i), C.byref(o), None) == nat.STE_ERR_INVALID_ARG  # null arrays
    assert native_lib.ste_sigma_points_f64(9, 1, 1, 1.0, None, None, None, None, None) == nat.STE_ERR_UNSUPPORTED
    with pytest.raises(nat.NativeError):
        nat.check(nat.STE_ERR_INVALID_ARG)


def test_no_cpu_fallback():
    """CPU tensors are refused by the binding; the product package never imports the oracle."""
    import torch

    from ship_track_estimators_b200 import _native as nat

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        nat.ptr(torch.zeros(4, dtype=torch.float64))
    pkg = os.path.join(REPO, "ship_track_estimators_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(root, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f
                assert "host_emul" not in text or f.endswith(".cuh"), f
