"""Cost of the innovation statistics on one GPU: the forward pass with and without the nis / loglik / rank planes
(``allocate(..., innovations=True)``), the two launches alternating in every repetition so that both see the same machine
state.  Prints one JSON line: per shape the median and min-max seconds of each form over the timed launches (after one
warm-up launch of each), the ratio of the medians, and the card's name, power limit and max SM clock.

    python tools/innovation_perf.py [--reps 7] [--out profiles/innovation_perf.json]

Shapes:
  c5   the bench.py config-5 tile: 151 552 tracks x 1 024 steps, k = 1, position-only update, packed covariances,
       long_steps=False, with the smoother's statistics tape as bench.py's forward pass writes it;
  c4   a config-4-shaped tile: 37 888 ragged tracks of 100-1 200 fixes, gaps of 1-24 h, k = 2, 1 % displaced fixes,
       Mahalanobis gating, packed covariances, long_steps=True (tools/config_perf.py's gated C4 shape);
  n5   the tools/fleet_n5_perf.py five-state tile: 151 552 ragged tracks of 129-257 fixes, k = 1, shared Q / R.
The planes share every other buffer with the run without them.  Needs a CUDA device: there is no CPU measurement."""
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


def with_planes(res, b):
    """A result set sharing ``res``'s buffers, plus innovation planes for tile ``b``."""
    from ship_track_estimators_b200.batch import allocate_innovations

    twin = type(res)(**{**res.__dict__})
    allocate_innovations(twin, b.max_obs, b.n_tracks, b.device)
    return twin


def measure(engine, b, res, reps):
    res_i = with_planes(res, b)
    t = time_alternating({"plain": lambda: engine.forward(b, res), "innovations": lambda: engine.forward(b, res_i)}, reps)
    torch.cuda.synchronize()
    same = bool(torch.equal(res.status, res_i.status))
    row = {"tracks": b.n_tracks, "track_steps": b.track_steps(), "status_equal": same}
    for name, (med, lo, hi) in t.items():
        row[name] = {"forward_s": med, "forward_min_max_s": [lo, hi], "track_steps_per_s": b.track_steps() / med}
    row["innovations_vs_plain"] = t["innovations"][0] / t["plain"][0]
    del res_i
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("innovation_perf needs a CUDA device")
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.synthetic import make_tracks

    out = {"gpu": gpu_info(), "reps": args.reps, "timing": "CUDA events around each forward launch; median and min-max"}
    H, Q, P = np.diag([1.0, 1.0, 0.0, 0.0]), np.diag([1e-2, 1e-2, 1e-4, 1e-4]), np.eye(4)

    ukf = BatchedUKF(H, Q, np.diag([1e-3, 1e-3, 0.0, 0.0]), P, packed_cov=True, long_steps=False)
    b = TrackBatch.from_synthetic(make_tracks(148 * 1024, 1025, seed=1000, device="cuda"), substeps=1)
    res = ukf.allocate(b, smoother=True)
    out["c5"] = measure(ukf, b, res, args.reps)
    del b, res
    torch.cuda.empty_cache()

    ukf = BatchedUKF(H, Q, np.diag([0.05, 0.05, 0.0, 0.0]), P, gating=True, packed_cov=True, long_steps=True)
    syn = make_tracks(148 * 128 * 2, 1200, seed=2, device="cuda", nobs_min=100, dts_choices=(1, 2, 3, 6, 12, 24), outlier_frac=0.01,
                      smooth_width=2)
    b = TrackBatch.from_synthetic(syn, 2, need_rows=ukf.model.rows_needed())
    del syn
    res = ukf.allocate(b, smoother=True)
    out["c4"] = measure(ukf, b, res, args.reps)
    del b, res
    torch.cuda.empty_cache()

    pad = lambda M, v: np.pad(M, ((0, 1), (0, 1))) + np.diag([0, 0, 0, 0, v])   # noqa: E731
    engine = BatchedUKFN(pad(H, 0.0), pad(Q, 1e-6), pad(np.diag([1e-3, 1e-3, 0.0, 0.0]), 0.0), pad(P, 1e-2))
    syn = make_tracks(151552, 257, seed=7, device="cuda", nobs_min=128, dts_choices=(1.0, 2.0, 3.0))
    b = TrackBatchN.from_batch(TrackBatch.from_synthetic(syn, substeps=1), turn_rate0=0.0)
    del syn
    res = engine.allocate(b, smoother=False)
    out["n5"] = measure(engine, b, res, args.reps)
    del b, res
    torch.cuda.empty_cache()

    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
