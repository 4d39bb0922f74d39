"""CPU: the C ABI of the device text formatter (exported, bound, argument checks that return before any launch), its
power-of-ten table, the exact conversion compiled for the host against CPython's '%.18e', and the formatter option."""
import ctypes as C
import os
import re
import subprocess
from fractions import Fraction

import numpy as np
import pytest

from _helpers import REPO

CSRC = os.path.join(REPO, "ship_track_estimators_b200", "csrc")


def test_text_symbols_are_exported_and_bound(native_lib):
    from ship_track_estimators_b200 import _native as nat

    text = open(os.path.join(REPO, "include", "ste_ukf.h")).read()
    assert int(re.search(r"#define STE_ABI_VERSION (\d+)", text).group(1)) == nat.STE_ABI_VERSION == native_lib.ste_version() == 7
    assert int(re.search(r"#define STE_TEXT_MAX_VALUE_BYTES (\d+)", text).group(1)) == nat.STE_TEXT_MAX_VALUE_BYTES
    for name in ("ste_text_convert_f64", "ste_text_write"):
        assert name in nat._PROTOTYPES and hasattr(native_lib, name)
    assert C.sizeof(nat.SteTextTable) == 72   # 3 x 8 B, 4 x 4 B, plane[8]


def _table(nat, **kw):
    t = nat.SteTextTable()
    t.base, t.track, t.ld, t.n_tracks, t.row_stride, t.row_div, t.n_cols = 0x1000, 0x2000, 8, 8, 4, 1, 4
    for c in range(4):
        t.plane[c] = c
    for k, v in kw.items():
        setattr(t, k, v)
    return t


@pytest.mark.parametrize("case", ["ok_empty", "null_tables", "null_base", "null_track", "ld", "neg_items", "neg_values", "plane_high",
                                  "plane_neg", "n_cols", "row_div", "n_tables", "null_outputs"])
def test_convert_argument_checks(case, native_lib):
    from ship_track_estimators_b200 import _native as nat

    table = {"null_base": _table(nat, base=None), "null_track": _table(nat, track=None), "ld": _table(nat, ld=7),
             "plane_high": _table(nat, plane=(C.c_int32 * 8)(0, 1, 2, 4)), "plane_neg": _table(nat, plane=(C.c_int32 * 8)(-1, 1, 2, 3)),
             "n_cols": _table(nat, n_cols=9), "row_div": _table(nat, row_div=0)}.get(case, _table(nat))
    arr = (nat.SteTextTable * 1)(table)
    n_tables = 9 if case == "n_tables" else 1
    n_items, n_values = (-1 if case == "neg_items" else 2), (-5 if case == "neg_values" else 0 if case == "ok_empty" else 10)
    outs = [None] * 3 if case == "null_outputs" else [0x3000, 0x4000, 0x5000]
    tables = None if case == "null_tables" else arr
    rc = native_lib.ste_text_convert_f64(tables, n_tables, n_items, 0x6000, n_values, *outs, None)
    if case == "ok_empty":
        assert rc == nat.STE_OK
    else:
        assert rc == nat.STE_ERR_INVALID_ARG, case
        assert native_lib.ste_last_error()


def test_write_argument_checks(native_lib):
    from ship_track_estimators_b200 import _native as nat

    w = native_lib.ste_text_write
    assert w(10, 0x1000, 0x2000, 0x3000, 0x4000, 27 * 10 - 1, None) == nat.STE_ERR_INVALID_ARG   # output too small
    assert b"STE_TEXT_MAX_VALUE_BYTES" in native_lib.ste_last_error()
    assert w(-1, 0x1000, 0x2000, 0x3000, 0x4000, 0, None) == nat.STE_ERR_INVALID_ARG
    assert w(10, None, 0x2000, 0x3000, 0x4000, 270, None) == nat.STE_ERR_INVALID_ARG
    assert w(10, 0x1000, 0x2000, 0x3000, None, 270, None) == nat.STE_ERR_INVALID_ARG
    assert w(0, 0x1000, 0x2000, 0x3000, 0x4000, 0, None) == nat.STE_OK


def test_power_of_ten_table_is_10_to_the_16j_in_106_bits():
    src = open(os.path.join(CSRC, "ste_text.cuh")).read()
    rows = re.findall(r"\{(-?0x[0-9a-f.p+-]+), (-?0x[0-9a-f.p+-]+), (-?\d+)\},\s*/\* 1e(-?\d+) \*/", src)
    assert [int(r[3]) for r in rows] == [16 * j for j in range(-19, 22)]
    for hi, lo, e2, p in rows:
        hi, lo, e2 = float.fromhex(hi), float.fromhex(lo), int(e2)
        assert 1.0 <= hi < 2.0
        exact = Fraction(10) ** int(p) / Fraction(2) ** e2
        assert hi == float(exact) and lo == float(exact - Fraction(hi))


def test_exact_conversion_on_the_host(tmp_path):
    """ste_text.cuh is __host__ __device__: compiled for the CPU it must already give CPython's strings."""
    from ship_track_estimators_b200 import build

    prog = tmp_path / "conv.cu"
    prog.write_text('#include "%s"\n#include <cstdio>\n' % os.path.join(CSRC, "ste_text.cuh") + r'''
int main(int argc, char **argv) {
    FILE *in = fopen(argv[1], "rb"), *out = fopen(argv[2], "wb");
    double x; char buf[32];
    while (fread(&x, 8, 1, in) == 1) {
        uint64_t d; int32_t m;
        ste::text::convert(x, d, m);
        const int n = ste::text::format_field(d, m | ste::text::kMetaNewline, buf);
        if (n != ste::text::field_length(m) + 1) return 1;
        fwrite(buf, 1, n, out);
    }
    return fclose(out) | fclose(in);
}
''')
    exe = str(tmp_path / "conv")
    subprocess.run([build._nvcc(), "-std=c++17", "-O2", "-o", exe, str(prog)], check=True, capture_output=True)
    rng = np.random.default_rng(7)
    m = rng.integers(1_600_000_000_000_000, 4_500_000_000_000_000, size=5000) * 2 + 1
    x = np.concatenate([rng.integers(0, 2**64, size=100_000, dtype=np.uint64).view(np.float64), m * 2.0 ** -5, -m * 2.0 ** -3,
                        [float(f"1e{k}") for k in range(-323, 309)], [np.nextafter(float(f"1e{k}"), 0) for k in range(-300, 309)],
                        [0.0, -0.0, np.inf, -np.inf, np.nan, 5e-324, np.finfo(np.float64).max]])
    x.astype(np.float64).tofile(tmp_path / "in.bin")
    subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.txt")], check=True)
    assert (tmp_path / "out.txt").read_text() == "".join("%.18e\n" % v for v in x)


def test_formatter_option(tmp_path):
    import torch

    from ship_track_estimators_b200.batch import TrackResults
    from ship_track_estimators_b200.cli import writers
    from ship_track_estimators_b200.ingest import FleetFixes

    fleet = FleetFixes(["1"], np.zeros((2, 1)), np.zeros((2, 1)), np.ones((1, 1)), np.array([2], dtype=np.int32))
    res = TrackResults(torch.zeros(2, 4, 1, dtype=torch.float64), torch.zeros(2, 16, 1, dtype=torch.float64), None, None,
                       torch.zeros(1, dtype=torch.int32), torch.zeros(1, dtype=torch.int32))
    with pytest.raises(ValueError, match="formatter"):
        writers.write_fleet_outputs("o", fleet, res, 1, str(tmp_path), formatter="gpu")
    with pytest.raises(ValueError, match='formatter="host"'):
        writers.write_fleet_outputs("o", fleet, res, 1, str(tmp_path), formatter="device")
    assert writers.write_fleet_outputs("o", fleet, res, 1, str(tmp_path), formatter="host") == 4
    settings = {"dim": 4, "H": [1.0] * 4, "R": [1e-3] * 4, "Q": [1e-2] * 4, "P": [1.0] * 4, "dt": -1, "nsteps": 1}
    with pytest.raises(ValueError, match="formatter"):
        writers.estimate_fleet(str(tmp_path / "missing.csv"), settings, device="cpu", formatter="text")


def test_table_rejects_host_and_strided_sources():
    import torch

    from ship_track_estimators_b200.text import Table

    track = torch.zeros(1, dtype=torch.int32)
    with pytest.raises(ValueError, match="contiguous CUDA"):
        Table(torch.zeros(3, 4, 2, dtype=torch.float64), track, [0]).native()
    with pytest.raises(ValueError, match="contiguous CUDA"):
        Table(torch.zeros(3, 4, 4, dtype=torch.float64)[:, :, :2], track, [0]).native()
