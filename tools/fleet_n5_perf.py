"""Five-state fleet path (geodetic_dynamics_turn, batch_n.BatchedUKFN) on one GPU: kernel times, track-steps/s, FP64
operations and HBM bytes per track-step counted from the shapes, the n = 4 BatchedUKF on the same tile for context, and
the class API's per-step cost.  Prints one JSON line.

    python tools/fleet_n5_perf.py [--tracks 151552] [--steps 256] [--reps 5] [--per-track-noise] [--out profiles/fleet_n5_perf.json]

The tile is ragged (make_tracks, lengths uniform in [steps/2, steps] fixes per track at k = 1, the same step count at
k = 2); its inputs and outputs (about 70 GB at the default size) are far above the 126 MB L2.  Needs a CUDA device: there
is no CPU measurement.

``--per-track-noise`` also runs the tile with its own Q and R per track (``TrackBatchN.Q`` / ``R``: two ship classes,
alternate tracks, differing in the position R and the turn-rate Q) and times it against the shared-matrix tile, the two
launches alternating in every repetition so that both see the same machine state."""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np
import torch


def fp64_flops_per_step(n=5, upd_fraction=1.0):
    """FP64 operations (an FMA counts 2) of one predict [+ update] and one backward step, counted from the loops of
    csrc/ste_generic.cuh for the fixed-size algebra.  Excluded: the Jacobi sweeps of the two square roots / two
    pseudo-inverses (data-dependent sweep count) and the trigonometry of the process model (11 evaluations per step)."""
    L = 2 * n + 1
    fun_sym = 2 * n * n + 3 * n ** 3               # symmetrise + V f V^T (a multiply and an FMA per term)
    predict = n * n + fun_sym + 2 * n * L + 2 * n * L + 5 * n * n * L + n * n
    update = 2 * n ** 3 * 2 + fun_sym + 2 * n ** 3 + 2 * 2 * n * n + 2 * n ** 3 * 3 + 4 * n ** 3
    backward = n * n + fun_sym + 2 * n * L + 2 * n * L + 2 * 5 * n * n * L + fun_sym + 2 * n ** 3 + 4 * n * n + 3 * n ** 3 + 2 * n ** 3
    return {"forward": predict + upd_fraction * update, "backward": backward}


def hbm_bytes_per_step(n=5, upd_fraction=1.0):
    """Algorithmic HBM traffic per track-step: the forward writes one filtered state (n + n*n doubles) and reads dt, the
    mask byte, two rate rows and, per update, n observation rows; the backward reads the filtered state and dt / rates
    and writes the smoothed state."""
    state = 8 * (n + n * n)
    return {"forward": state + 8 + 1 + 16 + upd_fraction * 8 * n, "backward": 2 * state + 8 + 16}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_launches(fn, reps):
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(times)), float(min(times)), float(max(times))


def time_alternating(fns, reps):
    """Median / min / max seconds of each launch in ``fns`` (name -> callable), the launches interleaved per repetition."""
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name in fns}
    for _ in range(reps):
        for name, fn in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            times[name].append(a.elapsed_time(b) * 1e-3)
    return {name: (float(np.median(t)), float(min(t)), float(max(t))) for name, t in times.items()}


def class_planes(T, Q, R):
    """[25][T] planes of two ship classes on alternate tracks: the given (Q, R), and a logbook class with R = 0.25 deg^2
    on the position and a 100x larger turn-rate Q."""
    Q2, R2 = Q.copy(), R.copy()
    Q2[4, 4] *= 100.0
    R2[0, 0] = R2[1, 1] = 0.25
    odd = (np.arange(T) % 2).astype(bool)
    planes = lambda A, B: torch.from_numpy(np.where(odd[None, :], B.reshape(25, 1), A.reshape(25, 1))).to("cuda")   # noqa: E731
    return planes(Q, Q2), planes(R, R2)


def fp64_peak():
    """DFMA throughput of this card measured by the library's probe (ste_probe_fp64_fma) - the compute ceiling used below."""
    from ship_track_estimators_b200 import _native as nat

    lib = nat.load()
    blocks, threads, iters = 148 * 16, 256, 20000
    sink = torch.empty(blocks * threads, dtype=torch.float64, device="cuda")
    run = lambda: nat.check(lib.ste_probe_fp64_fma(blocks, threads, iters, nat.ptr(sink), nat.current_stream()))   # noqa: E731
    med, _, _ = time_launches(run, 5)
    return 2 * 8 * iters * blocks * threads / med


def class_api(steps=1000):
    """Public predict + update at n = 5 (one launch and two copies each: the route run took before the fleet kernel), and
    run over one track of `steps` steps: the public-call loop against the one-launch run."""
    from types import SimpleNamespace

    from ship_track_estimators_b200.kalman_filters import UnscentedKalmanFilter, geodetic_dynamics_turn

    H = np.zeros((5, 5))
    H[:2, :2] = np.eye(2)
    Q, R = np.diag([1e-2, 1e-2, 1e-4, 1e-4, 1e-6]), np.diag([1e-3, 1e-3, 0.0, 0.0, 0.0])
    make = lambda: UnscentedKalmanFilter(H=H, Q=Q, R=R, P=np.eye(5), x0=np.array([10.0, 20.0, 15.0, 90.0, 0.1]),   # noqa: E731
                                         non_linear_process=geodetic_dynamics_turn, noise="zero")
    ukf, z = make(), np.array([10.1, 20.05, 15.0, 90.0, 0.0])
    for _ in range(20):
        ukf.predict(dt=1.0, c=None, sog_rate=0.0)
        ukf.update(z)
    torch.cuda.synchronize()
    n = 300
    t0 = time.perf_counter()
    for _ in range(n):
        ukf.predict(dt=1.0, c=None, sog_rate=0.0)
        ukf.update(z)
    torch.cuda.synchronize()
    per_step = (time.perf_counter() - t0) / n
    rng = np.random.default_rng(0)
    m = steps + 1
    zt = np.stack([10 + np.cumsum(rng.normal(size=m)) * 0.01, 20 + np.cumsum(rng.normal(size=m)) * 0.01, np.full(m, 15.0), np.full(m, 90.0)])
    tr = SimpleNamespace(dts=np.ones(steps), z=zt, sog_rate=np.zeros(m), cog_rate=np.zeros(m))
    u = make()
    u.run(steps, np.ones(steps), tr)
    t0 = time.perf_counter()
    u = make()
    u.run(steps, np.ones(steps), tr)
    run_after = time.perf_counter() - t0
    u = make()
    t0 = time.perf_counter()
    u.update(np.append(zt[:, 0], 0.0))
    for s in range(steps):   # the former route of run at n = 5: one predict and one update launch per step
        u.predict(dt=1.0, c=None, sog_rate=0.0)
        u.update(np.append(zt[:, s + 1], 0.0))
    torch.cuda.synchronize()
    run_before = time.perf_counter() - t0
    return {"predict_plus_update_us": per_step * 1e6, "run_1000_steps_s_before": run_before, "run_1000_steps_s_after": run_after}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=151552)
    ap.add_argument("--steps", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--per-track-noise", action="store_true", help="also time the tile with per-track Q and R")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fleet_n5_perf needs a CUDA device")
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.batch_n import BatchedUKFN, TrackBatchN
    from ship_track_estimators_b200.synthetic import make_tracks

    info = gpu_info()
    H4, Q4, R4 = np.diag([1.0, 1, 0, 0]), np.diag([1e-2, 1e-2, 1e-4, 1e-4]), np.diag([1e-3, 1e-3, 0, 0])
    pad = lambda M, v: np.pad(M, ((0, 1), (0, 1))) + np.diag([0, 0, 0, 0, v])   # noqa: E731
    engine = BatchedUKFN(pad(H4, 0.0), pad(Q4, 1e-6), pad(R4, 0.0), pad(np.eye(4), 1e-2))
    peak = fp64_peak()
    out = {"gpu": info, "tracks": args.tracks, "max_steps": args.steps, "block": int(os.environ.get("STE_N5_THREADS_LABEL", "64")),
           "fp64_dfma_probe_tflops": peak / 1e12, "hbm_datasheet_tbps": 7.7}
    for k in (1, 2):
        nobs = args.steps // k + 1
        syn = make_tracks(args.tracks, nobs, seed=7, device="cuda", nobs_min=nobs // 2, dts_choices=(1.0, 2.0, 3.0))
        b4 = TrackBatch.from_synthetic(syn, substeps=k)
        del syn
        b = TrackBatchN.from_batch(b4, turn_rate0=0.0)
        steps = b.track_steps()
        res = engine.allocate(b)
        if args.per_track_noise:
            Qp, Rp = class_planes(b.n_tracks, engine.Q, engine.R)
            bq = TrackBatchN(**{**b.__dict__, "Q": Qp, "R": Rp})
            resq = engine.allocate(bq)   # a result set of its own: the smoother reads the states its tile filtered
            fwd_all = time_alternating({"shared": lambda: engine.forward(b, res), "per_track": lambda: engine.forward(bq, resq)}, args.reps)
            bwd_all = time_alternating({"shared": lambda: engine.backward(b, res), "per_track": lambda: engine.backward(bq, resq)}, args.reps)
            st_q = resq.check_status(raise_on=0)
            del resq
            fwd, bwd = fwd_all["shared"], bwd_all["shared"]
        else:
            fwd = time_launches(lambda: engine.forward(b, res), args.reps)
            bwd = time_launches(lambda: engine.backward(b, res), args.reps)
        st = res.check_status(raise_on=0)
        del res
        torch.cuda.empty_cache()
        e4 = BatchedUKF(H4, Q4, R4, np.eye(4))
        r4 = e4.allocate(b4)
        n4 = time_launches(lambda: e4.run(b4, res=r4), args.reps)
        del r4
        torch.cuda.empty_cache()
        fl, by = fp64_flops_per_step(upd_fraction=1.0 / k), hbm_bytes_per_step(upd_fraction=1.0 / k)
        row = {"track_steps": steps, "status": st,
               "forward_s": fwd[0], "forward_min_max_s": fwd[1:], "backward_s": bwd[0], "backward_min_max_s": bwd[1:],
               "forward_track_steps_per_s": steps / fwd[0], "backward_track_steps_per_s": steps / bwd[0],
               "both_track_steps_per_s": steps / (fwd[0] + bwd[0]),
               "fp64_flops_per_track_step_counted": fl, "hbm_bytes_per_track_step": by}
        for p in ("forward", "backward"):
            t = row[f"{p}_s"]
            row[f"{p}_fp64_share_of_probe_peak"] = fl[p] * steps / t / peak
            row[f"{p}_hbm_share_of_datasheet"] = by[p] * steps / t / 7.7e12
        if args.per_track_noise:
            fq, bq_ = fwd_all["per_track"], bwd_all["per_track"]
            row["per_track_noise"] = {"status": st_q, "forward_s": fq[0], "forward_min_max_s": fq[1:], "backward_s": bq_[0],
                                      "backward_min_max_s": bq_[1:], "both_track_steps_per_s": steps / (fq[0] + bq_[0]),
                                      "forward_vs_shared": fq[0] / fwd[0], "backward_vs_shared": bq_[0] / bwd[0],
                                      "both_vs_shared": (fq[0] + bq_[0]) / (fwd[0] + bwd[0])}
            del bq, Qp, Rp
        row["n4_batched_ukf_run_s"] = n4[0]
        row["n4_batched_ukf_track_steps_per_s"] = steps / n4[0]
        out[f"k{k}"] = row
        del b, b4
        torch.cuda.empty_cache()
    out["class_api_n5"] = class_api()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
