"""Cost of per-track process noise on the n = 4 passes (``TrackBatch.Q``) on one GPU.  Three forms of each tile, their
launches alternating in every repetition so that all see the same machine state:
  shared   the tile as it is: the filter's Q for every track (the existing kernels);
  planes   the same tile with per-track planes that all hold the filter's Q: the arithmetic is the same, so this against
           ``shared`` is the cost of the per-track kernels alone (the tool asserts that every output is bit-identical);
  classes  two ship classes on alternate tracks with different Q.
The forward and the backward pass are timed separately (CUDA events around each launch, one warm-up launch of each form,
then the median and min-max of ``--reps``).  Prints one JSON line with the card's name, power limit and max SM clock.

    python tools/per_track_q_perf.py [--reps 5] [--out profiles/per_track_q_perf.json]

Tiles (those of tools/innovation_perf.py):
  c5   the bench.py config-5 tile: 151 552 tracks x 1 024 steps, k = 1, position-only update, packed covariances,
       long_steps=False, with the smoother's statistics tape;
  c4   a config-4-shaped tile: 37 888 ragged tracks of 100-1 200 fixes, gaps of 1-24 h, k = 2, 1 % displaced fixes,
       Mahalanobis gating, packed covariances, long_steps=True, with the tape.
Needs a CUDA device: there is no CPU measurement."""
import argparse
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import numpy as np
import torch

from fleet_n5_perf import gpu_info, time_alternating

Q_SHARED = np.diag([1e-2, 1e-2, 1e-4, 1e-4])
# a second ship class: larger, correlated position noise and correlated speed / course noise
Q_CLASS2 = np.array([[4e-2, 1e-2, 0.0, 0.0], [1e-2, 3e-2, 0.0, 0.0], [0.0, 0.0, 1e-3, 2e-4], [0.0, 0.0, 2e-4, 4e-3]])
OUTPUTS = ("mean_f", "cov_f", "mean_s", "cov_s", "status", "n_updates", "gate_iters", "gate_lambda", "gate_scale", "smooth_stats")


def planes(T, mats):
    """[16][T] planes on the device, track t holding mats[t % len(mats)]."""
    cols = np.stack([mats[t % len(mats)].reshape(-1) for t in range(T)], axis=1)
    return torch.from_numpy(np.ascontiguousarray(cols)).to("cuda")


def allocate(engine, b):
    res = engine.allocate(b, smoother=True)
    for name in ("mean_f", "cov_f", "mean_s", "cov_s", "smooth_stats"):   # rows past a ragged track's end compare too
        getattr(res, name).zero_()
    return res


def measure(engine, b, reps):
    from dataclasses import replace

    T = b.n_tracks
    tiles = {"shared": b, "planes": replace(b, Q=planes(T, [Q_SHARED])), "classes": replace(b, Q=planes(T, [Q_SHARED, Q_CLASS2]))}
    res = {name: allocate(engine, t) for name, t in tiles.items()}
    fwd = time_alternating({name: (lambda n=name: engine.forward(tiles[n], res[n])) for name in tiles}, reps)
    bwd = time_alternating({name: (lambda n=name: engine.backward(tiles[n], res[n])) for name in tiles}, reps)
    torch.cuda.synchronize()
    for name in OUTPUTS:
        x, y = getattr(res["shared"], name), getattr(res["planes"], name)
        if x is not None:   # bit patterns: the tape marks invalid entries with NaN
            bits = (lambda t: t.view(torch.int64)) if x.dtype == torch.float64 else (lambda t: t)
            assert torch.equal(bits(x), bits(y)), f"{name}: per-track planes holding the shared Q changed the output"
    steps = b.track_steps()
    row = {"tracks": T, "track_steps": steps, "planes_bit_identical": True,
           "classes_differ": not torch.equal(res["shared"].mean_s, res["classes"].mean_s)}
    for pas, t in (("forward", fwd), ("backward", bwd)):
        row[pas] = {name: {"s": med, "min_max_s": [lo, hi], "track_steps_per_s": steps / med} for name, (med, lo, hi) in t.items()}
        row[pas]["planes_vs_shared"] = t["planes"][0] / t["shared"][0]
        row[pas]["classes_vs_shared"] = t["classes"][0] / t["shared"][0]
    del res, tiles
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("per_track_q_perf needs a CUDA device")
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.synthetic import make_tracks

    out = {"gpu": gpu_info(), "reps": args.reps,
           "timing": "CUDA events around each launch, the three forms alternating; median and min-max after one warm-up each"}
    H, P = np.diag([1.0, 1.0, 0.0, 0.0]), np.eye(4)

    ukf = BatchedUKF(H, Q_SHARED, np.diag([1e-3, 1e-3, 0.0, 0.0]), P, packed_cov=True, long_steps=False)
    b = TrackBatch.from_synthetic(make_tracks(148 * 1024, 1025, seed=1000, device="cuda"), substeps=1)
    out["c5"] = measure(ukf, b, args.reps)
    del b
    torch.cuda.empty_cache()

    ukf = BatchedUKF(H, Q_SHARED, np.diag([0.05, 0.05, 0.0, 0.0]), P, gating=True, packed_cov=True, long_steps=True)
    syn = make_tracks(148 * 128 * 2, 1200, seed=2, device="cuda", nobs_min=100, dts_choices=(1, 2, 3, 6, 12, 24), outlier_frac=0.01,
                      smooth_width=2)
    b = TrackBatch.from_synthetic(syn, 2, need_rows=ukf.model.rows_needed())
    del syn
    out["c4"] = measure(ukf, b, args.reps)
    del b
    torch.cuda.empty_cache()

    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
