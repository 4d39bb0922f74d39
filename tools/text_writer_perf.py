"""Rate of the device text formatter (csrc/ste_text.cu) and wall time of write_fleet_outputs with each formatter.

    python tools/text_writer_perf.py [--values 33554432] [--ships 20000] [--host-ships 1000] [--out profiles/text_writer.json]

1. Kernels alone: convert + inclusive scan + write (text.format_tables), CUDA events over repeated passes, on
   (a) a mix of typical values (lon / lat, variances across 14 decades, step lengths) and (b) random 64-bit patterns.
2. write_fleet_outputs for an n = 4 and an n = 5 fleet of ragged ships (64-128 fixes, smoother on) into a temporary
   directory that is deleted afterwards: the device formatter on ``--ships`` ships (wall time split into format, device
   to host copy and file writes) and the host formatter (np.savetxt) on the first ``--host-ships`` of them.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from ship_track_estimators_b200.batch import BatchedUKF  # noqa: E402
from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN  # noqa: E402
from ship_track_estimators_b200.cli import writers  # noqa: E402
from ship_track_estimators_b200.cli.writers import write_fleet_outputs  # noqa: E402
from ship_track_estimators_b200.ingest import FleetFixes  # noqa: E402
from ship_track_estimators_b200.text import Table, format_tables  # noqa: E402


def kernel_rate(x: np.ndarray, reps: int = 10) -> dict:
    dev = torch.device("cuda")
    base = torch.from_numpy(x).to(dev).reshape(-1, 1, 1)
    n = base.shape[0]
    tables = [Table(base, torch.zeros(1, dtype=torch.int32, device=dev), [0])]
    vs = torch.tensor([0, n], dtype=torch.int64, device=dev)
    format_tables(tables, vs, n)                             # warm-up
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        _, off = format_tables(tables, vs, n)
    b.record()
    b.synchronize()
    s = a.elapsed_time(b) / 1e3 / reps
    return {"values": n, "seconds_per_pass": s, "values_per_s": n / s, "text_bytes": int(off[-1]), "text_GB_per_s": int(off[-1]) / s / 1e9}


def make_fleet(ships: int, seed: int) -> FleetFixes:
    rng = np.random.default_rng(seed)
    n_obs = rng.integers(64, 129, size=ships).astype(np.int32)
    m = int(n_obs.max())
    lon = np.cumsum(rng.normal(0, 0.02, (m, ships)), axis=0) + rng.uniform(-170, 170, ships)
    lat = np.cumsum(rng.normal(0, 0.02, (m, ships)), axis=0) + rng.uniform(-60, 60, ships)
    dts = rng.choice([0.5, 1.0, 2.0, 3.0], size=(m - 1, ships))
    rows = np.arange(m)[:, None]
    lon[rows >= n_obs], lat[rows >= n_obs] = 0.0, 0.0
    dts[rows[:-1] >= n_obs - 1] = 0.0
    return FleetFixes([str(200000000 + t) for t in range(ships)], lon, lat, dts, n_obs)


def fleet_times(dim: int, ships: int, host_ships: int, tmp: str) -> dict:
    fleet = make_fleet(ships, seed=dim)
    H, Q, R = np.diag([1.0, 1, 0, 0]), np.diag([1e-2, 1e-2, 1e-4, 1e-4]), np.diag([1e-3, 1e-3, 0, 0])
    if dim == 4:
        ukf = BatchedUKF(H, Q, R, np.eye(4))
        res = ukf.run(fleet.to_batch(device="cuda", substeps=1, need_rows=ukf.model.rows_needed()), smoother=True)
    else:
        d = np.diag
        ukf = BatchedUKFN(d([1.0, 1, 0, 0, 0]), d([1e-2, 1e-2, 1e-4, 1e-4, 1e-5]), d([1e-3, 1e-3, 0, 0, 0]), d([1.0, 1, 1, 4, 1e-2]))
        res = ukf.run(TrackBatchN.from_batch(fleet.to_batch(device="cuda", substeps=1, need_rows=(True,) * 4)), smoother=True)
    torch.cuda.synchronize()
    out = {"dim": dim, "ships": ships, "track_steps": int(fleet.n_obs.sum() - ships)}
    for label, formatter, sel in (("device", "device", None), ("host", "host", list(range(host_ships)))):
        d = os.path.join(tmp, f"{dim}_{label}")
        os.makedirs(d)
        stats = {}
        t0 = time.perf_counter()
        files = write_fleet_outputs("output", fleet, res, 1, d, ships=sel, formatter=formatter,
                                    stats=stats if formatter == "device" else None)
        wall = time.perf_counter() - t0
        n = ships if sel is None else len(sel)
        out[label] = dict(ships=n, files=files, wall_s=wall, ships_per_s=n / wall, files_per_s=files / wall, **stats)
        shutil.rmtree(d)
    dv = out["device"]
    # write_s sums the busy time of the writer threads
    dv["writer_threads"] = writers._WRITER_THREADS
    dv["write_thread_share"] = dv["write_s"] / (writers._WRITER_THREADS * dv["wall_s"])
    out["speedup_per_ship"] = dv["ships_per_s"] / out["host"]["ships_per_s"]
    out["speedup_note"] = (f"per-ship rates: the device formatter wrote all {ships} ships, the host formatter (np.savetxt) "
                           f"the first {host_ships}")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--values", type=int, default=1 << 25)
    ap.add_argument("--ships", type=int, default=20000)
    ap.add_argument("--host-ships", type=int, default=1000)
    ap.add_argument("--out", default="profiles/text_writer.json")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("text_writer_perf.py measures on a CUDA device; none is available")
    rng = np.random.default_rng(0)
    q = a.values // 4
    typical = np.concatenate([rng.uniform(-180, 180, q), rng.uniform(-90, 90, q), 10.0 ** rng.uniform(-12, 2, q),
                              rng.choice([0.5, 1.0, 2.0, 3.0], a.values - 3 * q) / 3.0])
    rng.shuffle(typical)
    bits = rng.integers(0, 2**64, size=a.values, dtype=np.uint64).view(np.float64)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip()
    res = {"gpu": smi, "kernels_typical": kernel_rate(typical), "kernels_random_bits": kernel_rate(bits)}
    with tempfile.TemporaryDirectory() as tmp:
        res["fleet_n4"] = fleet_times(4, a.ships, a.host_ships, tmp)
        res["fleet_n5"] = fleet_times(5, a.ships, a.host_ships, tmp)
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
