#!/usr/bin/env python
"""Every ship of a CSV at once: what the reference's batch example loops over ship by ship
(examples/example_ukf_rts_smoother_batch.py there) as one parse, one filter launch and one smoother launch.

    python examples/fleet_from_csv.py <tracks.csv> <input.json> [--out-dir results --id-col primary.id --device-parse]

Writes the CLI's five text files per ship (output_<id>_predictions.txt, ...) and prints a per-fleet summary.
An input.json with "dim": 5 (5 x 5 H, Q, R, P) runs the five-state turn-rate model (geodetic_dynamics_turn) instead.
"""
import argparse
import json
import os
import time

import torch

from ship_track_estimators_b200.cli.writers import estimate_fleet
from ship_track_estimators_b200.performance_metrics import track_metrics  # noqa: F401  (per-track fit metrics, see README)

ap = argparse.ArgumentParser()
ap.add_argument("csv")
ap.add_argument("settings", help="the CLI's input.json (dim, H, Q, R, P, dt, nsteps, smooth)")
ap.add_argument("--out-dir", default="results")
ap.add_argument("--id-col", default="primary.id")
ap.add_argument("--lat-col", default="lat")
ap.add_argument("--lon-col", default="lon")
ap.add_argument("--geodesy", default="wgs84", choices=["wgs84", "sphere"])
a = ap.parse_args()

os.makedirs(a.out_dir, exist_ok=True)
settings = json.load(open(a.settings))
t0 = time.perf_counter()
fleet, results = estimate_fleet(a.csv, settings, id_col=a.id_col, lat_col=a.lat_col, lon_col=a.lon_col, apply_rts_smoother=True,
                                output_prefix="output", directory=a.out_dir, geodesy=a.geodesy)
torch.cuda.synchronize()
dt = time.perf_counter() - t0
steps = int(results.n_steps_host.sum())
print(f"{fleet.n_tracks} ships, {int(fleet.n_obs.sum())} fixes, {steps} filter steps in {dt:.2f} s (parse, derive, filter, smooth, write)")
print(f"flagged tracks: {int((results.status != 0).sum())}; files in {a.out_dir}/")
