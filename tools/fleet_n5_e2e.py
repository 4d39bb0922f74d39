"""Five-state fleet path end to end on one GPU: pinned host tiles through ``BatchedUKFN.run_host_pipelined`` for each
output set (inputs host->device, forward + backward, the selected outputs device->host, on three overlapped streams),
and ``performance_metrics.track_metrics`` on a resident tile.  Prints one JSON line: track-steps/s and bytes moved per
direction for each output set, and the metrics kernel's time.

    python tools/fleet_n5_e2e.py [--tracks 151552] [--steps 128] [--tiles 4] [--out profiles/fleet_n5_e2e.json]

Tiles are ragged (make_tracks, lengths uniform in [steps/2, steps] fixes per track, k = 1), two distinct pinned input
tiles used alternately; results go to two pinned output sets used alternately, as a consumer that drains each set
before it comes round again would.  The "all" set of one default tile is 9.4 GB, far above the 126 MB L2.  Needs a
CUDA device: there is no CPU measurement."""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch

from fleet_n5_perf import gpu_info, time_launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=151552)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--tiles", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fleet_n5_e2e needs a CUDA device")
    from ship_track_estimators_b200.batch import TrackBatch
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.performance_metrics import track_metrics
    from ship_track_estimators_b200.synthetic import make_tracks

    H = np.zeros((5, 5))
    H[:2, :2] = np.eye(2)
    engine = BatchedUKFN(H, np.diag([1e-2, 1e-2, 1e-4, 1e-4, 1e-6]), np.diag([1e-3, 1e-3, 0.0, 0.0, 0.0]),
                         np.diag([1.0, 1.0, 1.0, 1.0, 1e-2]))
    nobs = args.steps + 1
    pinned = []
    for seed in (7, 8):
        syn = make_tracks(args.tracks, nobs, seed=seed, device="cuda", nobs_min=nobs // 2, dts_choices=(1.0, 2.0, 3.0))
        pinned.append(TrackBatchN.from_batch(TrackBatch.from_synthetic(syn, substeps=1)).pin_memory())
        del syn
    torch.cuda.empty_cache()
    host_tiles = [pinned[i % 2] for i in range(args.tiles)]
    steps = sum(t.track_steps() for t in host_tiles)
    out = {"gpu": gpu_info(), "tracks_per_tile": args.tracks, "max_steps": args.steps, "tiles": args.tiles, "track_steps": steps,
           "input_bytes_per_tile": pinned[0].input_bytes()}
    for name in engine.OUTPUT_SETS:
        sets = [engine.host_outputs(pinned[0], outputs=name) for _ in range(2)]
        host_outs = [sets[i % 2] for i in range(args.tiles)]
        engine.run_host_pipelined(host_tiles[:2], host_outs[:2], outputs=name)   # warm-up: buffers, streams, modules
        torch.cuda.synchronize()
        times = []
        for _ in range(2):
            t0 = time.perf_counter()
            moved = engine.run_host_pipelined(host_tiles, host_outs, outputs=name)
            torch.cuda.synchronize()
            times.append(time.perf_counter() - t0)
        t = min(times)
        out[name] = {"s": t, "s_runs": times, "track_steps_per_s": steps / t, "h2d_bytes": moved["h2d_bytes"],
                     "d2h_bytes": moved["d2h_bytes"], "h2d_gb_per_s": moved["h2d_bytes"] / t / 1e9,
                     "d2h_gb_per_s": moved["d2h_bytes"] / t / 1e9,
                     "d2h_bytes_per_stored_state": moved["d2h_bytes"] / (args.tiles * args.tracks * (args.steps + 1))}
        del sets, host_outs
        engine._pipe = None
        torch.cuda.empty_cache()
    # resident tile: the two passes, then the metrics kernel on the filtered and the smoothed states
    b = pinned[0].to("cuda")
    res = engine.run(b)
    torch.cuda.synchronize()
    run = time_launches(lambda: engine.run(b, res=res), args.reps)
    out["resident_run_s"], out["resident_track_steps_per_s"] = run[0], b.track_steps() / run[0]
    for which in ("filtered", "smoothed"):
        m = time_launches(lambda: track_metrics(engine, b, res, which=which), args.reps)
        out[f"metrics_{which}_s"] = m[0]
        out[f"metrics_{which}_min_max_s"] = m[1:]
    out["status"] = res.check_status(raise_on=0)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
