"""Scoring 32 noise candidates on one GPU: one ``score`` call (the store-free scoring launch, all candidates in one
launch per update variant) against the route it replaces - 32 forward passes with innovation planes, one engine per
candidate, the result buffers allocated once and reused.  The two forms alternate in every repetition so that both see the
same machine state.  Prints one JSON line: per shape the median and min-max seconds of each form over the timed
repetitions (after one warm-up of each), the ratio of the medians, the device memory each form needs beyond the tile's
inputs, whether the two forms agree, and the card's name, power limit and max SM clock.

    python tools/noise_score_perf.py [--reps 5] [--out profiles/noise_score_perf.json]

Shapes (those of tools/innovation_perf.py, plus a small fleet):
  c5     151 552 tracks x 1 024 steps, k = 1, position-only update, packed covariances, long_steps=False;
  c4     37 888 ragged tracks of 100-1 200 fixes, gaps of 1-24 h, k = 2, 1 % displaced fixes, gating, packed covariances,
         long_steps=True;
  n5     151 552 ragged five-state tracks of 129-257 fixes, k = 1;
  small  2 048 tracks x 1 024 steps, otherwise as c5: one candidate fills 16 of 148 SMs.
The candidates are noise_grid(Q, R, (0.5, 1, 2, 4), (0.25, 0.5, 1, 2, 4, 8, 16, 32)).  Needs a CUDA device."""
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

Q_SCALES, R_SCALES = (0.5, 1.0, 2.0, 4.0), (0.25, 0.5, 1.0, 2.0, 4.0, 8.0, 16.0, 32.0)


def nbytes(tensors):
    return int(sum(t.numel() * t.element_size() for t in tensors if t is not None))


def measure(make_engine, b, cands, reps):
    """(a) one score call; (b) one forward pass with innovation planes per candidate into shared result buffers."""
    from ship_track_estimators_b200.performance_metrics import innovation_metrics

    engines = [make_engine(Q, R) for Q, R in cands]
    res = engines[0].allocate(b, smoother=False, innovations=True)
    out = {}

    def score():
        out["score"] = engines[0].score(b, cands)

    def forwards():
        sums = []
        for e in engines:
            e.forward(b, res)
            sums.append(innovation_metrics(res)["loglik"])
        out["forwards"] = sums

    t = time_alternating({"score": score, "forwards": forwards}, reps)
    torch.cuda.synchronize()
    got, ref = out["score"]["loglik"], torch.stack(out["forwards"])
    finite = torch.isfinite(ref) & torch.isfinite(got)
    rel = float(((got - ref).abs() / ref.abs().clamp(min=1.0))[finite].max()) if bool(finite.any()) else 0.0
    row = {"tracks": b.n_tracks, "track_steps": b.track_steps(), "candidates": len(cands),
           "score_vs_forwards_max_rel_diff_loglik": rel,   # the forwards' sums are torch reductions, not update order
           "same_nonfinite": bool(torch.equal(torch.isfinite(ref), torch.isfinite(got))),
           "input_bytes": b.input_bytes(),
           "score_output_bytes": nbytes(out["score"].values()),
           "forwards_buffer_bytes": nbytes([getattr(res, n) for n in res._TENSORS])}
    for name, (med, lo, hi) in t.items():
        row[name] = {"seconds": med, "min_max_seconds": [lo, hi],
                     "candidate_track_steps_per_s": len(cands) * b.track_steps() / med}
    row["score_vs_forwards"] = t["score"][0] / t["forwards"][0]
    del res, engines, out
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--shapes", default="c5,c4,n5,small")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("noise_score_perf needs a CUDA device")
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.synthetic import make_tracks
    from ship_track_estimators_b200.tuning import noise_grid

    shapes = args.shapes.split(",")
    out = {"gpu": gpu_info(), "reps": args.reps,
           "timing": "CUDA events around each form; median and min-max over the repetitions, the two forms alternating",
           "shapes": {}}
    H, Q, P = np.diag([1.0, 1.0, 0.0, 0.0]), np.diag([1e-2, 1e-2, 1e-4, 1e-4]), np.eye(4)
    R_pos = np.diag([1e-3, 1e-3, 0.0, 0.0])

    for name, T in (("c5", 148 * 1024), ("small", 2048)):
        if name not in shapes:
            continue
        b = TrackBatch.from_synthetic(make_tracks(T, 1025, seed=1000, device="cuda"), substeps=1)
        make = lambda Qc, Rc: BatchedUKF(H, Qc, Rc, P, packed_cov=True, long_steps=False)   # noqa: E731
        out["shapes"][name] = measure(make, b, noise_grid(Q, R_pos, Q_SCALES, R_SCALES), args.reps)
        del b
        torch.cuda.empty_cache()

    if "c4" in shapes:
        R_gate = np.diag([0.05, 0.05, 0.0, 0.0])
        make = lambda Qc, Rc: BatchedUKF(H, Qc, Rc, P, gating=True, packed_cov=True, long_steps=True)   # noqa: E731
        syn = make_tracks(148 * 128 * 2, 1200, seed=2, device="cuda", nobs_min=100, dts_choices=(1, 2, 3, 6, 12, 24), outlier_frac=0.01,
                          smooth_width=2)
        b = TrackBatch.from_synthetic(syn, 2, need_rows=make(Q, R_gate).model.rows_needed())
        del syn
        out["shapes"]["c4"] = measure(make, b, noise_grid(Q, R_gate, Q_SCALES, R_SCALES), args.reps)
        del b
        torch.cuda.empty_cache()

    if "n5" in shapes:
        pad = lambda M, v: np.pad(M, ((0, 1), (0, 1))) + np.diag([0, 0, 0, 0, v])   # noqa: E731
        H5, Q5, R5, P5 = pad(H, 0.0), pad(Q, 1e-6), pad(R_pos, 0.0), pad(P, 1e-2)
        syn = make_tracks(151552, 257, seed=7, device="cuda", nobs_min=128, dts_choices=(1.0, 2.0, 3.0))
        b = TrackBatchN.from_batch(TrackBatch.from_synthetic(syn, substeps=1), turn_rate0=0.0)
        del syn
        out["shapes"]["n5"] = measure(lambda Qc, Rc: BatchedUKFN(H5, Qc, Rc, P5), b, noise_grid(Q5, R5, Q_SCALES, R_SCALES), args.reps)
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
