#!/usr/bin/env python
"""Benchmark of the fp64 UKF + URTSS hot path on synthetic ship tracks (BASELINE.json configs 3-5).

    python bench.py [--config c5|c3|c4] [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

``--config c5`` (default; BASELINE.json configs[4], the one the metric is quoted on): 16 M tracks x
1024 steps, constant dt = 1 h, k = 1, UKF + URTSS, zero noise, track-sharded over the GPUs.  16 M
tracks do not fit one GPU's HBM at once (inputs alone are 690 GB), so the job runs as tiles of
``--tracks`` tracks; a "step" of the benchmark is one pass of the hot path (forward filter +
backward smoother) over one tile whose inputs are already resident in HBM.  Per-GPU work is fixed
as N grows (weak scaling) and there is no collective inside the timed region.  The line also
carries ``job``: the WHOLE 16 M-track job pushed through the tile loop (this rank's
``sharding.shard_range`` share, per-tile ``track_metrics``, one final NCCL summary), wall-clocked.

``--config c3`` (configs[2]): 1 M x 1024, forward filter only.  ``--config c4`` (configs[3]): 1 M
ragged tracks of 100-5000 fixes, gaps drawn from {1,2,3,6,12,24} h, k = 2 sub-steps, box smoothing
2, 1 % displaced fixes, Mahalanobis gating + URTSS, processed as length-sorted tiles
(``sharding.plan_ragged_tiles``, dealt round-robin to the ranks).

One JSON line is printed by rank 0; see README / DESIGN.md for the keys.  ``--dump-outputs DIR`` also writes the
results of the last timed step (a seeded sample of its tracks) as ``DIR/*.npy``: the inputs are seeded, so two builds
run with the same arguments can be compared output for output.  ``--impl reference``
times the reference's own CPU implementation of the same path (the unmodified reference installed
under ``baseline/_ref`` when present, else the numpy oracle port) on all host cores of the box.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

MODEL = dict(H=[1.0, 1.0, 0.0, 0.0], R=[1e-3, 1e-3, 0.0, 0.0], Q=[1e-2, 1e-2, 1e-4, 1e-4], P=[1.0, 1.0, 1.0, 1.0])
UNIT = "track-steps/s"
GRANULE = 148 * 128   # one block of 128 tracks per SM

CONFIGS = {
    "c5": dict(workload="configs[4]: synthetic 16M tracks x 1024 steps UKF+URTSS fp64, track-sharded; processed in resident tiles",
               metric="track-steps/sec (UKF+URTSS fp64)", n_steps=1024, k=1, smoother=True, gating=False, ragged=False,
               job_tracks=16 * 1024 * 1024, scaling="weak", e2e_outputs="smoothed"),
    "c2": dict(workload="configs[1]: the batch example's fleet on one B200 - the 71 runnable ships of data/historical_ships and one ship of "
                        "data/modern_ships, inputs exactly as the reference's ShipTrack derives them (committed with the reference's own "
                        "outputs in tests/golden/c2_*.npz), dt=-1, nsteps=2 sub-steps, UKF+URTSS; two resident tiles (one per model)",
               metric="track-steps/sec (UKF+URTSS fp64, the reference's ship data)", k=2, smoother=True, gating=False, ragged=True,
               fleet=("c2_historical_batch", "c2_modern_ship"), job_tracks=72, scaling="strong", e2e_outputs="smoothed"),
    "c3": dict(workload="configs[2]: synthetic 1M tracks x 1024 steps, constant dt=1, fp64 UKF forward filter only; processed in resident tiles",
               metric="track-steps/sec (UKF forward fp64)", n_steps=1024, k=1, smoother=False, gating=False, ragged=False,
               job_tracks=1024 * 1024, scaling="weak", e2e_outputs="filtered"),
    "c4": dict(workload="configs[3]: synthetic 1M ragged tracks (100-5000 obs), gaps in {1,2,3,6,12,24} h, k=2 sub-steps, smooth=2, "
                        "1% displaced fixes, Mahalanobis robustification + URTSS; length-sorted tiles",
               metric="track-steps/sec (gated UKF+URTSS fp64, ragged)", k=2, smoother=True, gating=True, ragged=True,
               nobs_min=100, nobs_max=5000, dts_choices=(1.0, 2.0, 3.0, 6.0, 12.0, 24.0), outlier_frac=0.01, smooth_width=2,
               job_tracks=1024 * 1024, scaling="strong", e2e_outputs="smoothed"),
}


def alg_bytes(k, smoother):
    """Algorithmic bytes per track-step (SURVEY.md 8(d)): forward 168 + 32/k, backward 328 + 16/k."""
    fwd, bwd = 168.0 + 32.0 / k, 328.0 + 16.0 / k
    return fwd, (bwd if smoother else 0.0)


def kernel_counts(shape="uniform"):
    """Instruction / flop / DRAM-byte counts per track-step of the kernels, written from ncu captures by
    tools/ncu_counts.py (profiles/kernel_counts.json: the uniform k = 1 shape of configs 3 / 5) and
    tools/c4_counts.py (profiles/kernel_counts_c4.json: the ragged, gated k = 2 shape of config 4); None when absent."""
    path = os.path.join(REPO, "profiles", "kernel_counts.json" if shape == "uniform" else "kernel_counts_c4.json")
    if os.path.exists(path):
        with open(path) as fh:
            return json.load(fh)
    return None


def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_cores() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def np_model():
    import numpy as np

    return tuple(np.diag(MODEL[k]) for k in ("H", "R", "Q", "P"))


# ------------------------------------------------------------------------------------------- #
# CPU arm: the reference (or its oracle port) on host cores                                   #
# ------------------------------------------------------------------------------------------- #
def load_fleet(names):
    """The committed real-data fixtures (tests/golden/*.npz, written by tests/golden/make_golden.py from the reference's data
    files and its own outputs): -> list of per-ship dicts (inputs H, Q, R, P0, x0, z, dts, dt_array, rates; reference means / covs)."""
    import numpy as np

    ships = []
    for name in names:
        d = np.load(os.path.join(REPO, "tests", "golden", name + ".npz"), allow_pickle=False)
        n = int(d["n_tracks"])
        group = [dict(fixture=name) for _ in range(n)]
        for key in d.files:
            head, _, tail = key.partition("_")
            if head.startswith("t") and head[1:].isdigit():
                group[int(head[1:])][tail] = d[key]
        ships += group
    return ships


def _cpu_worker_fleet(job):
    """Worker c of C: ships c, c + C, ... of the fleet through the reference (or the numpy port)."""
    kind, cfg_name, index, stride = job
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"
    import numpy as np

    ships = load_fleet(CONFIGS[cfg_name]["fleet"])[index::stride]
    if kind == "reference":
        from oracle import reference_arm as RA
        RA.load()
    else:
        from oracle import ukf_numpy as O
    t0 = time.perf_counter()
    done = 0
    for sh in ships:
        k = len(sh["dt_array"]) // len(sh["dts"])
        if kind == "reference":
            RA.run_track(sh["z"], sh["dts"], k, sh["H"], sh["Q"], sh["R"], sh["P0"], sh["sog_rate"], sh["cog_rate"], smoother=True)
        else:
            O.run_track(sh["x0"], sh["P0"], sh["H"], sh["Q"], sh["R"], sh["dt_array"], sh["dts"], sh["z"], sh["sog_rate"], sh["cog_rate"], smoother=True)
        done += len(sh["dt_array"])
    return done, time.perf_counter() - t0


def _cpu_sample(cfg_name, seed, n_tracks):
    """Synthetic tracks of the config's shape for the CPU arms (generated with the same generator
    as the GPU tiles).  The ragged config is sampled at a bounded length (its mean is 2550 fixes)."""
    from ship_track_estimators_b200.synthetic import make_tracks

    cfg = CONFIGS[cfg_name]
    if cfg["ragged"]:
        return make_tracks(n_tracks, 640, seed=seed, device="cpu", nobs_min=384, dts_choices=cfg["dts_choices"],
                           outlier_frac=cfg["outlier_frac"], smooth_width=cfg["smooth_width"])
    return make_tracks(n_tracks, cfg["n_steps"] + 1, seed=seed, device="cpu")


def _cpu_worker(job):
    """One worker = one core: a few synthetic tracks through the reference's run / run_rts_smoother
    (kind "reference") or through the numpy oracle port (kind "port")."""
    kind, cfg_name, seed, n_tracks = job
    for var in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[var] = "1"
    import numpy as np

    import scipy.linalg  # noqa: F401  (imported once per worker by the warm-up job)
    import torch  # noqa: F401

    if n_tracks == 0:
        return 0, 0.0
    cfg = CONFIGS[cfg_name]
    syn = _cpu_sample(cfg_name, seed, n_tracks)
    H, R, Q, P = np_model()
    if kind == "reference":
        from oracle import reference_arm as RA
        RA.load()
    else:
        from oracle import ukf_numpy as O
    t0 = time.perf_counter()
    done = 0
    for t in range(n_tracks):
        m = int(syn.nobs[t])
        z = np.stack([syn.lon[:m, t].numpy(), syn.lat[:m, t].numpy(), syn.sog[:m, t].numpy(), syn.cog[:m, t].numpy()])
        dts = syn.dts[: m - 1, t].numpy()
        sr, cr = syn.sog_rate[:m, t].numpy(), syn.cog_rate[:m, t].numpy()
        if kind == "reference":
            RA.run_track(z, dts, cfg["k"], H, Q, R, P, sr, cr, smoother=cfg["smoother"], gating=cfg["gating"])
        else:
            O.run_track(z[:, 0], P, H, Q, R, O.generate_dts(dts, cfg["k"]), dts, z, sr, cr, smoother=cfg["smoother"], gating=cfg["gating"])
        done += (m - 1) * cfg["k"]
    return done, time.perf_counter() - t0


def _cpu_worker_c(job):
    """Uniform tracks through the plain-C oracle (oracle/ukf_oracle.c), one process per core."""
    _, cfg_name, seed, n_tracks = job
    from oracle import ukf_c as OC

    cfg = CONFIGS[cfg_name]
    syn = _cpu_sample(cfg_name, seed, n_tracks)
    H, R, Q, P = np_model()
    args = (syn.x0().numpy(), syn.dts.numpy(), syn.lon.numpy(), syn.lat.numpy(), syn.sog_rate.numpy(), syn.cog_rate.numpy(), H, Q, R, P)
    OC.load()
    t0 = time.perf_counter()
    OC.run_batch(*args, substeps=cfg["k"], smoother=cfg["smoother"])
    return n_tracks * cfg["n_steps"] * cfg["k"], time.perf_counter() - t0


def reference_kind() -> str:
    from oracle import reference_arm as RA

    return "reference" if RA.locate() else "port"


class CpuPool:
    """One spawned process per host core, each running the CPU implementation single-threaded."""

    def __init__(self, cores: int, kind: str, cfg_name: str):
        import multiprocessing as mp

        self.cores, self.kind, self.cfg_name = cores, kind, cfg_name
        self.pool = mp.get_context("spawn").Pool(cores)
        self.pool.map(_cpu_worker, [("port", "c5", 0, 0)] * cores)  # import numpy/scipy/torch once per worker

    def run(self, tracks_per_core: int, seed: int, worker=None):
        """-> (aggregate track-steps/s, track-steps done, slowest worker's busy seconds)."""
        jobs = [(self.kind, self.cfg_name, seed + c, tracks_per_core) for c in range(self.cores)]
        out = self.pool.map(worker or _cpu_worker, jobs, chunksize=1)
        steps, busy = sum(o[0] for o in out), max(o[1] for o in out)
        return steps / busy, steps, busy

    def run_fleet(self):
        """The whole fleet of a real-data config once, its ships dealt to the cores."""
        jobs = [(self.kind, self.cfg_name, c, self.cores) for c in range(self.cores)]
        out = self.pool.map(_cpu_worker_fleet, jobs, chunksize=1)
        steps, busy = sum(o[0] for o in out), max(o[1] for o in out)
        return steps / busy, steps, busy

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_sample_text(kind, cfg_name, cores, tracks_per_core, steps, busy):
    cfg = CONFIGS[cfg_name]
    what = {"reference": "the UNMODIFIED reference (baseline/_ref: UnscentedKalmanFilter.run"
                         + (" + run_rts_smoother" if cfg["smoother"] else "") + ", np.random.normal pinned to zero"
                         + (", robustification line re-enabled by a subclass" if cfg["gating"] else "") + ")",
            "port": "numpy oracle port calling the reference's own scipy.linalg.sqrtm / numpy.linalg.pinv"}[kind]
    if cfg.get("fleet"):
        return (f"the whole fleet once ({cfg['job_tracks']} ships, dealt to {cores} single-threaded processes), zero noise; {what}: "
                f"{steps} track-steps, slowest worker {busy:.1f} s")
    shape = "384-640 fixes, k=2 (bounded-length sample of the ragged shape)" if cfg["ragged"] else f"{cfg['n_steps']} steps"
    return (f"{cores} single-threaded processes x {tracks_per_core} track(s) x {shape} of the same synthetic workload, zero noise; {what}: "
            f"{steps} track-steps, slowest worker {busy:.1f} s")


# tracks per core and bench step of the reference arm: 4 x 1 024 steps are ~2 s per step on a B200 box's host cores (one
# track per step under-reads the reference by a third: the slowest of 16 workers over 0.4 s decides the step)
REF_ARM_TRACKS_PER_CORE = 4


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    cores, kind = host_cores(), reference_kind()
    pool = CpuPool(cores, kind, args.config)
    done = []
    for i in range(args.warmup + args.steps):
        _, steps, busy = pool.run_fleet() if cfg.get("fleet") else pool.run(REF_ARM_TRACKS_PER_CORE, seed=100 + 1000 * i)
        if i >= args.warmup:
            done.append((steps, busy))
    pool.close()
    value = sum(s for s, _ in done) / sum(b for _, b in done)
    line = {
        "impl": "reference", "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * statistics.mean(b for _, b in done), "higher_is_better": True,
        "scaling": cfg["scaling"], "vs_baseline": None, "dtype": "f64",
        "data": "synthetic" if not cfg.get("fleet") else "the reference's ship data (fixtures generated from data/historical_ships and "
                                                         "data/modern_ships by the unmodified reference)",
        # the same config block as the GPU arm prints for these arguments (the tile size names the GPU arm's resident
        # tile; the CPU sample of each step is described under cpu_baseline.sample)
        "config": workload_config(args, per_gpu_tracks=None if cfg["ragged"] else args.tracks),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "per_core": value / cores,
                         "sample": "each bench step = " + cpu_sample_text(kind, args.config, cores, 1 if cfg.get("fleet") else REF_ARM_TRACKS_PER_CORE, done[-1][0], done[-1][1])},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------- #
# helpers                                                                                     #
# ------------------------------------------------------------------------------------------- #
def workload_config(args, per_gpu_tracks):
    cfg = CONFIGS[args.config]
    out = {
        "workload": cfg["workload"], "config": args.config, "substeps": cfg["k"], "noise": "zero",
        "tile_tracks_per_gpu": per_gpu_tracks, "job_tracks": cfg["job_tracks"],
        "H": MODEL["H"], "R": MODEL["R"], "Q": MODEL["Q"], "P0": MODEL["P"],
        "cache": "inputs+outputs per step are GBs (>> 126 MB L2); input tiles alternate",
        "cov_storage": "full16" if getattr(args, "full_cov", False) else "packed10 (symmetric 4x4 stored as its 10 unique entries)",
        "parallelism": f"tracks sharded over {args.gpus} GPU(s), no data-path collective",
    }
    if cfg.get("fleet"):
        out.update(H="per fixture (H = diag(1,1,0,0))", R="per fixture (historical ships 0.25 deg^2, modern ship 1e-3)", Q="per fixture",
                   P0="identity", cache="the fleet's states fit the L2: a 256 MB buffer is overwritten between timed steps",
                   fixtures=list(cfg["fleet"]))
    elif cfg["ragged"]:
        out.update(nobs=[cfg["nobs_min"], cfg["nobs_max"]], dts_hours=list(cfg["dts_choices"]), smooth=cfg["smooth_width"],
                   outlier_frac=cfg["outlier_frac"], gating_chi=50.0)
    else:
        out.update(steps_per_track=cfg["n_steps"], dt_hours=1.0)
    return out


# --dump-outputs: a fixed, seeded sample of the track columns of the last timed step's results, at most this many bytes
DUMP_BYTES = 60 * 1000 * 1000
DUMP_SEED = 20251020


def sample_results(res, budget=DUMP_BYTES, prefix=""):
    """Host float64 copies of every result array of a TrackResults (its kernels' layout, tracks last), restricted to a
    seeded sample of track columns sized to ``budget`` bytes; ``<prefix>columns`` holds the sampled column indices."""
    import numpy as np
    import torch

    arrays, seen = {}, set()
    for name in res._TENSORS:
        t = getattr(res, name)
        if t is None or t.data_ptr() in seen:      # smoothed in place: mean_s / cov_s are mean_f / cov_f
            continue
        seen.add(t.data_ptr())
        arrays[name] = t
    T = res.status.shape[0]
    per_track = 8 * sum(t.numel() // T for t in arrays.values()) + 8
    n = min(T, budget // per_track)
    cols = np.sort(np.random.default_rng(DUMP_SEED).choice(T, size=n, replace=False))
    idx = torch.from_numpy(cols).to(res.status.device)
    out = {prefix + "columns": cols.astype(np.float64)}
    for name, t in arrays.items():
        a = t.index_select(t.dim() - 1, idx).to(torch.float64).cpu().numpy()
        if name in ("mean_f", "cov_f", "mean_s", "cov_s") and res.n_steps_host is not None:
            past = np.arange(a.shape[0])[:, None] > res.n_steps_host[cols][None, :]   # past a ragged track's end: never written
            a = np.where(past[:, None, :], 0.0, a)
        out[prefix + name] = a
    return out


def write_dump(directory, arrays):
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (one background
    `nvidia-smi -lms 50` process, read when the region ends)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            time.sleep(0.25)  # let the first samples arrive before the timed region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is None:
            return
        time.sleep(0.1)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=10)
        except Exception:
            self.proc.kill()
            out = ""
        self.rows = [[c.strip() for c in line.split(",")] for line in out.splitlines() if line.strip()]

    def summary(self):
        sm, reasons, mx = [], set(), None
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            try:
                clk, mx_ = float(r[0]), float(r[1])
            except (ValueError, IndexError):
                continue
            mx = mx_
            if clk < 0.5 * mx_:   # idle samples before / after the kernels
                continue
            sm.append(clk)
            for name, flag in zip(names, r[3:7]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples_under_load": len(sm), "samples": len(self.rows)}


class Dist:
    """torch.distributed plumbing of the bench: barrier, max / sum over ranks (NCCL)."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus and self.world == 1 and args.gpus > 1:
            raise SystemExit("launch multi-GPU runs with torchrun (one rank per GPU)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, value: float, op: str) -> float:
        if self.world == 1:
            return float(value)
        t = self.torch.tensor([value], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def fp64_probe(lib, nat, torch, dev):
    """DFMA peak of this GPU (TFLOP/s) from the library's dependent-free FMA probe."""
    blocks, threads, iters = 148 * 16, 256, 20000
    sink = torch.empty(blocks * threads, dtype=torch.float64, device=dev)
    nat.check(lib.ste_probe_fp64_fma(blocks, threads, 200, nat.ptr(sink), nat.current_stream()))
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    nat.check(lib.ste_probe_fp64_fma(blocks, threads, iters, nat.ptr(sink), nat.current_stream()))
    p1.record()
    torch.cuda.synchronize()
    return 2.0 * 8 * iters * blocks * threads / (p0.elapsed_time(p1) * 1e-3) / 1e12


def roofline_block(cfg, track_steps_per_launch, f_ms, b_ms, fp64_peak, full_cov):
    """`roofline` object of the JSON line: the dominant kernel against the measured HBM peak
    (algorithmic bytes), both kernels, the whole step, and the FP64-pipe view from the counted
    instructions (profiles/kernel_counts.json)."""
    peak, peak_src = measured_peaks()
    bytes_f, bytes_b = alg_bytes(cfg["k"], cfg["smoother"])
    # counts per shape: the ragged, gated config runs other instruction paths (full-range geodetic tier, 2-4 Jacobi sweeps per
    # root, gating) and has its own capture; the real-data fleet (72 tracks, latency-bound) has none
    counts = {} if cfg.get("fleet") else (kernel_counts("c4" if cfg["ragged"] else "uniform") or {})
    fwd_key = "forward" if cfg["smoother"] else "forward_no_tape"
    per_kernel = {}
    for key, ckey, alg, ms in (("forward", fwd_key, bytes_f, f_ms), ("backward", "backward", bytes_b, b_ms)):
        if ms is None or ms <= 0.0:
            continue
        gbs = alg * track_steps_per_launch / (ms * 1e-3) / 1e9
        per_kernel[key] = {"ms": ms, "algorithmic_bytes_per_track_step": alg, "algorithmic_gbs": gbs, "frac": gbs / peak}
        c = counts.get(ckey) or {}
        dram = c.get("dram_bytes_full_cov" if full_cov else "dram_bytes")
        if dram:
            dg = dram * track_steps_per_launch / (ms * 1e-3) / 1e9
            per_kernel[key].update(dram_bytes_per_track_step=dram, dram_gbs=dg, dram_frac=dg / peak)
        if c.get("fp64_rf_cycles"):   # pipe + register-file bound: sum of max(2, distinct register sources) over the FP64 instructions
            bound_ms = c["fp64_rf_cycles"] * track_steps_per_launch / 32.0 / (592 * 1.965e9) * 1e3
            per_kernel[key].update(fp64_rf_bound_ms=bound_ms, frac_of_fp64_rf_bound=bound_ms / ms)
        if c.get("fp64_instr"):
            per_kernel[key].update(
                fp64_instr_per_track_step=c["fp64_instr"], flops_per_track_step=c.get("flops"),
                tflops=(c.get("flops") or 0.0) * track_steps_per_launch / (ms * 1e-3) / 1e12,
                fp64_pipe_busy=c["fp64_instr"] * track_steps_per_launch / 32.0 * 2.05 / (ms * 1e-3 * 592 * 1.965e9))
    dom = max(per_kernel, key=lambda k: per_kernel[k]["ms"])
    d = per_kernel[dom]
    total_ms = sum(v["ms"] for v in per_kernel.values())
    step_gbs = (bytes_f + bytes_b) * track_steps_per_launch / (total_ms * 1e-3) / 1e9
    traffic = d.get("dram_bytes_per_track_step")
    return {
        "bound": "hbm", "kernel": {"forward": "ukf_forward_kernel", "backward": "urtss_backward_kernel"}[dom],
        "achieved": d["algorithmic_gbs"], "peak": peak, "unit": "GB/s", "frac": d["frac"],
        "traffic": traffic * track_steps_per_launch if traffic else None, "traffic_source": counts.get("source") or "not captured for this shape",
        "peak_source": peak_src, "algorithmic_bytes_per_track_step": d["algorithmic_bytes_per_track_step"],
        "kernel_ms": d["ms"], "kernels": per_kernel,
        "whole_step": {"achieved": step_gbs, "frac": step_gbs / peak, "algorithmic_bytes_per_track_step": bytes_f + bytes_b},
        "fp64_pipe": {"peak_tflops_measured": fp64_peak,
                      "note": "flops = 2*DFMA + DMUL + DADD and fp64_instr = DFMA + DMUL + DADD + DSETP warp-instructions per track-step, "
                              "counted with ncu (profiles/kernel_counts.json); peak = DFMA probe (ste_probe_fp64_fma); fp64_pipe_busy = "
                              "fp64_instr x 2.05 cycles issue interval over 592 sub-partitions at 1965 MHz; fp64_rf_bound = the same instructions at "
                              "max(2, distinct 64-bit register sources) cycles each (measured: a three-register DFMA issues every 3.0 cycles; "
                              "tools/fp64_operand_model.py, profiles/r02_fp64_issue_intervals.txt)"},
    }


def cpu_baseline_block(args, cfg_name):
    """The reference's CPU path on the box's host cores, a bounded sample (rank 0, N = 1 only)."""
    cores, kind = host_cores(), reference_kind()
    cfg = CONFIGS[cfg_name]
    pool = CpuPool(cores, kind, cfg_name)
    per_core = args.cpu_tracks_per_core if not cfg["ragged"] else max(1, args.cpu_tracks_per_core // 2)
    if cfg.get("fleet"):
        v, steps, busy = pool.run_fleet()
        pool.close()
        return {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "per_core": v / cores,
                "sample": cpu_sample_text(kind, cfg_name, cores, 0, steps, busy)}, None
    v, steps, busy = pool.run(per_core, seed=4321)
    block = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "per_core": v / cores,
             "sample": cpu_sample_text(kind, cfg_name, cores, per_core, steps, busy)}
    compiled = None
    if not cfg["ragged"]:
        vc, steps_c, busy_c = pool.run(64 * args.cpu_tracks_per_core, seed=8765, worker=_cpu_worker_c)
        compiled = {"value": vc, "unit": UNIT, "cores": cores, "per_core": vc / cores, "kind": "port",
                    "sample": (f"plain-C restatement (oracle/ukf_oracle.c, gcc -O2, one process per core): "
                               f"{steps_c} track-steps, slowest worker {busy_c:.1f} s")}
    pool.close()
    job_steps = cfg["job_tracks"] * (cfg["n_steps"] if not cfg["ragged"] else (cfg["nobs_min"] + cfg["nobs_max"]) // 2 * cfg["k"])
    block["job_extrapolation"] = {
        "labelled": "EXTRAPOLATION from the sample above, not a measurement",
        "job_track_steps": job_steps, "core_seconds": job_steps / (v / cores), "hours_on_this_box": job_steps / v / 3600.0}
    return block, compiled


# ------------------------------------------------------------------------------------------- #
# GPU arm, uniform tiles (configs 3 and 5)                                                     #
# ------------------------------------------------------------------------------------------- #
def run_uniform(args, D):
    import numpy as np
    import torch

    from ship_track_estimators_b200 import _native as nat
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.performance_metrics import track_metrics
    from ship_track_estimators_b200.sharding import reduce_summary, shard_range
    from ship_track_estimators_b200.synthetic import make_tracks

    cfg = CONFIGS[args.config]
    N, smoother = cfg["n_steps"], cfg["smoother"]
    dev, rank, world = D.dev, D.rank, D.world
    lib = nat.load()  # raises if the CUDA library is missing: no fallback
    H, R, Q, P = np_model()
    ukf = BatchedUKF(H, Q, R, P, packed_cov=not args.full_cov, long_steps=False)   # 5-60 km/h x 1 h: every step is short
    T = args.tracks

    # two resident input tiles (different seeds per rank and per tile) and one set of output buffers
    tiles = []
    for j in range(2):
        syn = make_tracks(T, N + 1, seed=1000 + 17 * rank + j, device=str(dev))
        tiles.append(TrackBatch.from_synthetic(syn, substeps=1))
        del syn
    res = ukf.allocate(tiles[0], smoother=smoother, in_place=args.in_place)
    torch.cuda.synchronize()
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def step(i, record):
        b = tiles[i % 2]
        marks = [ev() for _ in range(3)] if record else None
        if record:
            marks[0].record()
        ukf.forward(b, res)
        if record:
            marks[1].record()
        if smoother:
            ukf.backward(b, res)
        if record:
            marks[2].record()
        return marks

    for i in range(args.warmup):
        step(i, False)
    D.barrier()
    with ClockSampler(D.local_rank) as clocks:
        t_start, t_end = ev(), ev()
        t_start.record()
        marks = [step(args.warmup + i, True) for i in range(args.steps)]
        t_end.record()
        D.barrier()
    if args.dump_outputs and rank == 0:   # before the passes below reuse the buffers
        write_dump(args.dump_outputs, sample_results(res))
    total_ms = D.reduce(t_start.elapsed_time(t_end), "max")
    f_ms = statistics.mean(m[0].elapsed_time(m[1]) for m in marks)
    b_ms = statistics.mean(m[1].elapsed_time(m[2]) for m in marks) if smoother else None
    tile_steps = T * N
    value = world * tile_steps * args.steps / (total_ms * 1e-3)
    launches = (2 if smoother else 1) * args.steps

    # ---- the same K steps with the two passes of successive tiles on disjoint SMs ---- #
    partitioned = run_partitioned(args, D, ukf, tiles, res, f_ms + b_ms, tile_steps) if (smoother and not args.no_partitioned) else None

    # ---- the whole job through the tile loop ---- #
    job = None
    if not args.no_job:
        lo, hi = shard_range(cfg["job_tracks"], rank, world)
        mine = hi - lo
        n_full, rest = divmod(mine, T)
        partial = None
        if rest:   # the last, narrower tile of this rank's share (contiguous copies; set up before the clock starts)
            src = tiles[n_full % 2]
            partial = src._map(lambda t: t[..., :rest].contiguous())
            partial.n_steps_host = None if src.n_steps_host is None else src.n_steps_host[:rest]
            partial_res = ukf.allocate(partial, smoother=smoother, in_place=args.in_place)
        which = "smoothed" if smoother else "filtered"
        acc = torch.zeros(4, dtype=torch.float64, device=dev)      # sum over tracks of the per-track rmse, per state row
        flagged = torch.zeros((), dtype=torch.int64, device=dev)
        D.barrier()
        w0 = time.perf_counter()
        j0, j1 = ev(), ev()
        j0.record()
        for i in range(n_full + (1 if rest else 0)):
            b, r = (tiles[i % 2], res) if i < n_full else (partial, partial_res)
            ukf.forward(b, r)
            if smoother:
                ukf.backward(b, r)
            m = track_metrics(ukf, b, r, which=which)
            acc += torch.nan_to_num(m["rmse"]).sum(dim=1)
            flagged += (r.status & ~nat.STE_STATUS_SMOOTH_RECOMPUTE != 0).sum()
        j1.record()
        local = {"tracks": float(mine), "track_steps": float(mine) * N, "flagged": float(flagged.item()),
                 **{f"sum_rmse_{n}": float(v) for n, v in zip(("lon", "lat", "sog", "cog"), acc.tolist())}}
        summary = reduce_summary(local, device=dev)      # the job's only collective (NCCL all_reduce of 7 doubles)
        D.barrier()
        wall = D.reduce(time.perf_counter() - w0, "max")
        dev_s = D.reduce(j0.elapsed_time(j1) * 1e-3, "max")
        job = {"tracks": int(summary["tracks"]), "track_steps": summary["track_steps"], "tiles_per_gpu": n_full + (1 if rest else 0),
               "wall_s": wall, "device_s": dev_s, "value": summary["track_steps"] / wall, "unit": UNIT,
               "per_tile": "forward" + (" + backward" if smoother else "") + f" + track_metrics({which}) + on-device accumulation; one NCCL all_reduce at the end",
               "inputs": "two resident seeded tiles per GPU, alternating (16 M distinct tracks would be 690 GB of inputs); every tile's "
                         "filtering, smoothing and metrics are executed in full",
               "mean_rmse_deg": {n: summary[f"sum_rmse_{n}"] / summary["tracks"] for n in ("lon", "lat")},
               "flagged_tracks": int(summary["flagged"])}
        launches_job = (3 if smoother else 2) * (n_full + (1 if rest else 0))
        job["gpu_launches"] = launches_job
        if partial is not None:
            del partial, partial_res

    # ---- end-to-end through the public API with HOST buffers ---- #
    e2e = run_e2e(args, D, ukf, cfg, lambda j: TrackBatch.from_synthetic(
        make_tracks(args.e2e_tracks, N + 1, seed=5000 + 31 * rank + j, device=str(dev)), substeps=1), args.e2e_tracks * N)

    if rank == 0:
        line = base_line(args, cfg, value, world, total_ms / args.steps, T)
        line["roofline"] = roofline_block(cfg, tile_steps, f_ms, b_ms, fp64_probe(lib, nat, torch, dev), args.full_cov)
        line["roofline"]["forward_ms"], line["roofline"]["backward_ms"] = f_ms, b_ms
        line["e2e"], line["gpu_launches"], line["clocks"] = e2e, launches, clocks.summary()
        if job:
            line["job"] = job
        if partitioned:
            line["partitioned_schedule"] = partitioned
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"], compiled = cpu_baseline_block(args, args.config)
            if compiled:
                line["compiled_port"] = compiled
        print(json.dumps(line), flush=True)


def run_partitioned(args, D, ukf, tiles, res, back_to_back_ms, tile_steps):
    """K steady-state steps of the software-pipelined schedule: forward(tile i+1) on one set of SMs beside backward(tile i)
    on the rest (green contexts, ship_track_estimators_b200/partition.py).  Every timed step is one full forward and one full
    backward launch, as in the headline loop; the first tile is filtered before the clock starts and the last one smoothed
    after it stops.  An extra key: the headline `value` stays the two launches back to back on all SMs."""
    import torch

    from ship_track_estimators_b200.partition import SmPartition

    res2 = part = None
    try:
        free, _ = torch.cuda.mem_get_info(D.dev)
        need = sum(t.numel() * t.element_size() for t in vars(res).values() if isinstance(t, torch.Tensor))
        if free < 1.1 * need:
            raise MemoryError(f"a second result set needs {need / 1e9:.0f} GB, {free / 1e9:.0f} GB free")
        part = SmPartition(D.dev, smoother_sms=args.smoother_sms)
        res2 = ukf.allocate(tiles[0], smoother=True, in_place=args.in_place)
        sets = [res, res2]
        cur, fs, bs = torch.cuda.current_stream(D.dev), part.filter_stream, part.smoother_stream

        def stage(i, fwd=True, bwd=True, after=None):
            # forward(tile i) into sets[i % 2] beside backward(tile i - 1) from sets[(i - 1) % 2]; `after`: the event
            # pair (forward done, backward done) of the previous stage, which both of this stage's launches wait for
            if after:
                fs.wait_event(after[0]); fs.wait_event(after[1]); bs.wait_event(after[0]); bs.wait_event(after[1])
            done = [torch.cuda.Event(), torch.cuda.Event()]
            with torch.cuda.stream(fs):
                if fwd:
                    ukf.forward(tiles[i % 2], sets[i % 2])
                done[0].record(fs)
            with torch.cuda.stream(bs):
                if bwd:
                    ukf.backward(tiles[(i - 1) % 2], sets[(i - 1) % 2])
                done[1].record(bs)
            return done

        def run(k):
            fs.wait_stream(cur); bs.wait_stream(cur)
            ev = stage(0, bwd=False)                       # prime: tile 0 filtered
            for i in range(1, 3):
                ev = stage(i, after=ev)                    # warm the pipeline
            cur.wait_event(ev[0]); cur.wait_event(ev[1])
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(cur)
            fs.wait_event(t0); bs.wait_event(t0)
            for i in range(3, 3 + k):
                ev = stage(i, after=ev)
            cur.wait_event(ev[0]); cur.wait_event(ev[1])
            t1.record(cur)
            ev = stage(3 + k, fwd=False, after=ev)         # drain: the last tile smoothed
            cur.wait_event(ev[1])
            torch.cuda.synchronize(D.dev)
            return t0.elapsed_time(t1)

        run(1)
        local_ms, info = run(args.steps), {"filter_sms": part.filter_sms, "smoother_sms": part.smoother_sms}
    except Exception as exc:   # an extra measurement must not take the bench line with it
        local_ms, info = None, {"unavailable": f"{type(exc).__name__}: {exc}"}
    finally:
        del res2
        if part is not None:
            try:
                torch.cuda.synchronize(D.dev)
                part.close()
            except Exception:
                pass
    # the collectives are unconditional: a rank that could not measure must not leave the others waiting
    n_ok = D.reduce(0.0 if local_ms is None else 1.0, "sum")
    ms = D.reduce(local_ms or 0.0, "max")
    if n_ok < D.world:
        return info if "unavailable" in info else {"unavailable": "another rank could not measure it"}
    return {**_partitioned_line(D, tile_steps, args.steps, ms, back_to_back_ms), **info}


def _partitioned_line(D, tile_steps, steps, ms, back_to_back_ms):
    return {"value": D.world * tile_steps * steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
            "back_to_back_ms_per_step": back_to_back_ms, "gain": back_to_back_ms / (ms / steps), "steps": steps,
            "schedule": "forward(tile i+1) on the filter SMs beside backward(tile i) on the smoother SMs (CUDA green contexts); "
                        "the same two kernels, bit-identical results (tests/test_gpu_parity.py::test_partitioned_schedule_is_bit_identical); "
                        "BatchedUKF.run_many(partition=SmPartition(...))",
            "gpu_launches": 2 * steps}


def base_line(args, cfg, value, world, ms_per_step, tile_tracks):
    return {"metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, tile_tracks)}


def run_e2e(args, D, ukf, cfg, make_tile, tile_track_steps):
    """Same metric through BatchedUKF.run_host_pipelined: pinned HOST inputs -> device, forward
    (+ backward), the selected outputs -> pinned host, tile after tile with the copy engines
    overlapped with the kernels.  The headline set is the config's product (the smoothed track and
    its variances; filtered for the forward-only config); the other sets are timed beside it."""
    import torch

    dev, world, smoother = D.dev, D.world, cfg["smoother"]
    host_tiles = [make_tile(j).pin_memory() for j in range(2)]
    torch.cuda.empty_cache()
    n_tiles = max(4, min(args.steps, 6))
    seq_in = [host_tiles[i % 2] for i in range(n_tiles)]
    sets = [cfg["e2e_outputs"]]
    # the other output sets are timed beside the headline on one GPU only: under torchrun every rank would pin
    # several GB more of the one host's memory for numbers that do not enter the scaling run
    if not args.e2e_headline_only and world == 1:   # ragged tiles are tens of GB of pinned memory per full output set: headline + summary only
        sets += [s for s in (("summary",) if cfg["ragged"] else ("all", "cli", "summary")) if smoother]
    out, by_set = None, {}
    for name in sets:
        host_outs = [ukf.host_outputs(host_tiles[0], outputs=name, smoother=smoother) for _ in range(2)]
        seq_out = [host_outs[i % 2] for i in range(n_tiles)]
        ukf.run_host_pipelined(seq_in[:2], seq_out[:2], smoother=smoother, device=dev, outputs=name)  # warm-up
        passes = []
        for _ in range(3):   # three timed passes, the median is reported: the host side of PCIe is shared with other tenants
            D.barrier()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            moved = ukf.run_host_pipelined(seq_in, seq_out, smoother=smoother, device=dev, outputs=name)
            t1.record()
            D.barrier()
            passes.append(D.reduce(t0.elapsed_time(t1), "max"))
        ms = statistics.median(passes)
        v = world * tile_track_steps * n_tiles / (ms * 1e-3)
        first = next(iter(host_outs[0].values()))
        assert bool(torch.isfinite(first.double()).all()) and float(first.double().abs().sum()) > 0.0
        entry = {"value": v, "unit": UNIT, "h2d_bytes_per_step": moved["h2d_bytes"] // n_tiles, "d2h_bytes_per_step": moved["d2h_bytes"] // n_tiles,
                 "outputs": list(ukf.OUTPUT_SETS[name]), "passes_ms": passes}
        by_set[name] = entry
        if out is None:
            out = dict(entry, output_set=name, tile_tracks=host_tiles[0].n_tracks, steps=n_tiles,
                       api="BatchedUKF.run_host_pipelined (H2D, kernels and D2H of successive tiles overlap on three streams)")
        del host_outs, seq_out
        torch.cuda.empty_cache()
    out["by_output_set"] = by_set
    return out


# ------------------------------------------------------------------------------------------- #
# GPU arm, ragged fleet (config 4)                                                             #
# ------------------------------------------------------------------------------------------- #
def run_ragged(args, D):
    import numpy as np
    import torch

    from ship_track_estimators_b200 import _native as nat
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch
    from ship_track_estimators_b200.sharding import plan_ragged_tiles, reduce_summary, shard_tiles_round_robin
    from ship_track_estimators_b200.synthetic import make_tracks

    cfg = CONFIGS[args.config]
    k, dev, rank, world = cfg["k"], D.dev, D.rank, D.world
    lib = nat.load()
    H, R, Q, P = np_model()
    # long_steps=None: the tier of the geodetic step is chosen per tile from its own legs (no user knob)
    ukf = BatchedUKF(H, Q, R, P, gating=cfg["gating"], packed_cov=not args.full_cov)
    need = ukf.model.rows_needed()

    # the fleet: 1 M lengths drawn once (seeded), sorted by decreasing length, cut into tiles by a
    # budget of stored states, dealt round-robin to the ranks
    rng = np.random.default_rng(2024)
    nobs_all = np.sort(rng.integers(cfg["nobs_min"], cfg["nobs_max"] + 1, size=cfg["job_tracks"]))[::-1].astype(np.int32)
    plan = plan_ragged_tiles((nobs_all.astype(np.int64) - 1) * k, state_budget=args.state_budget, granule=GRANULE)
    mine = shard_tiles_round_robin(len(plan), rank, world)
    # all of this rank's tiles (--full-job), or K of them evenly spaced through the sorted fleet after W warm-up tiles
    def spaced(n, count):
        return [min(n - 1, int((i + 0.5) * n / count)) for i in range(count)] if n and count else []

    if args.full_job:
        pick, n_warm = list(mine), 0
    else:
        warm = [mine[i] for i in spaced(len(mine), args.warmup)]
        pick, n_warm = warm + [mine[i] for i in spaced(len(mine), args.steps)], len(warm)   # more steps than tiles: tiles repeat
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def make_tile(ti):
        lo, hi = plan[ti]
        lengths = torch.from_numpy(nobs_all[lo:hi].copy())
        syn = make_tracks(hi - lo, int(lengths.max()), seed=7000 + ti, device=str(dev), dts_choices=cfg["dts_choices"],
                          outlier_frac=cfg["outlier_frac"], smooth_width=cfg["smooth_width"], lengths=lengths)
        return TrackBatch.from_synthetic(syn, substeps=k, need_rows=need)

    recs, gated, flagged, long_tiles = [], 0, 0, 0
    D.barrier()
    with ClockSampler(D.local_rank) as clocks:
        for n, ti in enumerate(pick):
            b = make_tile(ti)                                    # untimed: input generation on the device
            r = ukf.allocate(b, smoother=True, in_place=True)    # smoothed states overwrite the filtered ones (memory)
            long_tiles += int(ukf._long_steps_for(b))            # (cached per tile; decided before the clock starts)
            torch.cuda.synchronize()
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            ukf.forward(b, r)
            e1.record()
            ukf.backward(b, r)
            e2.record()
            torch.cuda.synchronize()
            if n >= n_warm:
                recs.append((b.track_steps(), e0.elapsed_time(e1), e1.elapsed_time(e2), b.n_tracks, b.max_steps))
                gated += int((r.gate_iters > 0).sum())
                flagged += int(((r.status & ~nat.STE_STATUS_SMOOTH_RECOMPUTE) != 0).sum())
            if args.dump_outputs and rank == 0 and n == len(pick) - 1:
                write_dump(args.dump_outputs, sample_results(r))
            del b, r
            torch.cuda.empty_cache()
        D.barrier()
    steps_local = float(sum(x[0] for x in recs))
    f_ms, b_ms = sum(x[1] for x in recs), sum(x[2] for x in recs)
    total_ms = D.reduce(f_ms + b_ms, "max")
    summary = reduce_summary({"track_steps": steps_local, "tracks": float(sum(x[3] for x in recs)), "gated_updates": float(gated),
                              "flagged": float(flagged)}, device=dev)
    value = summary["track_steps"] / (total_ms * 1e-3)

    # end to end: one mid-fleet tile shape through the host-buffer API
    mid = mine[len(mine) // 2]
    lo, hi = plan[mid]
    hi = min(hi, lo + max(128, args.e2e_tracks // 4))
    lengths = torch.from_numpy(nobs_all[lo:hi].copy())

    def e2e_tile(j):
        syn = make_tracks(hi - lo, int(lengths.max()), seed=9000 + 13 * rank + j, device=str(dev), dts_choices=cfg["dts_choices"],
                          outlier_frac=cfg["outlier_frac"], smooth_width=cfg["smooth_width"], lengths=lengths)
        return TrackBatch.from_synthetic(syn, substeps=k, need_rows=need)

    e2e = run_e2e(args, D, ukf, cfg, e2e_tile, int((lengths.to(torch.int64) - 1).sum()) * k)

    if rank == 0:
        line = base_line(args, cfg, value, world, total_ms / max(len(recs), 1), None)
        line["steps"], line["warmup"] = len(recs), n_warm
        line["config"].update(
            tiling=f"sharding.plan_ragged_tiles: {len(plan)} tiles of the length-sorted fleet (state budget {args.state_budget:.3g}, "
                   f"widths {min(h - l for l, h in plan)}-{max(h - l for l, h in plan)} tracks), dealt round-robin to {world} rank(s)",
            timed="a 'step' is one tile: forward + backward timed with CUDA events per tile, inputs generated on the device between "
                  "tiles (untimed); value = track-steps of the timed tiles / sum of their device times (max over ranks)",
            tiles_timed=[{"tracks": x[3], "max_steps": x[4], "track_steps": x[0], "forward_ms": x[1], "backward_ms": x[2]} for x in recs],
            full_job=bool(args.full_job), smoothing="in place", long_steps_tiles=f"{long_tiles} of {len(pick)} tiles pinned to the full-range geodetic tier (automatic)")
        line["roofline"] = roofline_block(cfg, steps_local, f_ms, b_ms, fp64_probe(lib, nat, torch, dev), args.full_cov)
        line["roofline"]["forward_ms"], line["roofline"]["backward_ms"] = f_ms, b_ms
        line["e2e"], line["gpu_launches"], line["clocks"] = e2e, 2 * len(recs), clocks.summary()
        line["summary"] = summary
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"], _ = cpu_baseline_block(args, args.config)
        print(json.dumps(line), flush=True)


def run_fleet(args, D):
    """BASELINE configs[1]: the reference's batch example (examples/example_ukf_rts_smoother_batch.py:19-90) - one filter + smoother per
    ship in a Python loop there, one resident tile per model here.  A step = forward + backward over the whole fleet.  The fleet is
    small (72 ships, ~7 000 track-steps): the number it gives is launch- and latency-bound, which is what a user of the example sees."""
    from types import SimpleNamespace

    import numpy as np
    import torch

    from ship_track_estimators_b200 import _native as nat
    from ship_track_estimators_b200.batch import BatchedUKF, TrackBatch

    cfg = CONFIGS[args.config]
    dev, rank, world = D.dev, D.rank, D.world
    lib = nat.load()
    ships = load_fleet(cfg["fleet"])[rank::world]   # strong scaling: the ships dealt to the ranks
    groups = {}
    for sh in ships:
        groups.setdefault(sh["fixture"], []).append(sh)
    tiles, worst = [], 0.0
    for name, group in groups.items():
        g0 = group[0]
        ukf = BatchedUKF(g0["H"], g0["Q"], g0["R"], g0["P0"], packed_cov=not args.full_cov)
        sts = [SimpleNamespace(dts=sh["dts"], z=sh["z"], sog_rate=sh["sog_rate"], cog_rate=sh["cog_rate"]) for sh in group]
        host = TrackBatch.from_tracks(sts, [sh["dt_array"] for sh in group], device="cpu", x0=[sh["x0"] for sh in group])
        b = host.to(dev)
        tiles.append((ukf, b, ukf.allocate(b, smoother=True), group, host))
    flush = torch.empty(256 * 1024 * 1024 // 8, dtype=torch.float64, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    recs = []
    D.barrier()
    if True:
        for i in range(args.warmup + args.steps):
            flush.fill_(float(i))      # the fleet's states (a few MB) would otherwise stay in the 126 MB L2 between steps
            torch.cuda.synchronize()
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            for ukf, b, r, _, _ in tiles:
                ukf.forward(b, r)
            e1.record()
            for ukf, b, r, _, _ in tiles:
                ukf.backward(b, r)
            e2.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                recs.append((e0.elapsed_time(e1), e1.elapsed_time(e2)))
        D.barrier()
    # the model tiles are independent: each tile's forward + backward chain on its own stream (what the value is quoted on;
    # the pass above, one launch after the other, gives the forward / backward split)
    streams = [torch.cuda.Stream(device=dev) for _ in tiles]
    conc = []
    D.barrier()
    with ClockSampler(D.local_rank) as clocks:
        for i in range(args.warmup + args.steps):
            flush.fill_(float(-i))
            torch.cuda.synchronize()
            e0, e1 = ev(), ev()
            e0.record()
            for st_, (ukf, b, r, _, _) in zip(streams, tiles):
                st_.wait_event(e0)
                with torch.cuda.stream(st_):
                    ukf.forward(b, r)
                    ukf.backward(b, r)
                torch.cuda.current_stream().wait_stream(st_)
            e1.record()
            torch.cuda.synchronize()
            if i >= args.warmup:
                conc.append(e0.elapsed_time(e1))
        D.barrier()
    if args.dump_outputs and rank == 0:
        for _, _, r, group, _ in tiles:
            write_dump(args.dump_outputs, sample_results(r, DUMP_BYTES // len(tiles), prefix=group[0]["fixture"] + "_"))
    # parity against the reference's own outputs stored with the inputs (what tests/test_gpu_golden.py asserts)
    for ukf, b, r, group, _ in tiles:
        r.check_status()
        for i, sh in enumerate(group):
            got = r.track(i)
            d = got["means_s"] - sh["means_s"].reshape(got["means_s"].shape)
            d[:, 3] = (d[:, 3] + 180.0) % 360.0 - 180.0
            worst = max(worst, float(np.max(np.abs(d) / np.maximum(1.0, np.abs(sh["means_s"].reshape(d.shape))))))
    steps_local = float(sum(len(sh["dt_array"]) for sh in ships))
    f_ms, b_ms = sum(x[0] for x in recs), sum(x[1] for x in recs)
    total_ms = D.reduce(sum(conc), "max")
    steps_all = D.reduce(steps_local, "sum")
    value = steps_all * len(conc) / (total_ms * 1e-3)

    # end to end: the same tiles from pinned host memory, smoothed tracks and variances back to pinned host memory
    e2e_ms, moved_in, moved_out = [], 0, 0
    pinned = [(ukf, host.pin_memory(), ukf.host_outputs(host, outputs=cfg["e2e_outputs"], smoother=True)) for ukf, _, _, _, host in tiles]
    for i in range(3 + args.steps):
        D.barrier()
        t0, t1 = ev(), ev()
        t0.record()
        moved_in = moved_out = 0
        for ukf, host, outs in pinned:
            moved = ukf.run_host_pipelined([host], [outs], smoother=True, device=dev, outputs=cfg["e2e_outputs"])
            moved_in, moved_out = moved_in + moved["h2d_bytes"], moved_out + moved["d2h_bytes"]
        t1.record()
        torch.cuda.synchronize()
        D.barrier()
        if i >= 3:
            e2e_ms.append(D.reduce(t0.elapsed_time(t1), "max"))
    e2e = {"value": steps_all / (statistics.median(e2e_ms) * 1e-3), "unit": UNIT, "h2d_bytes_per_step": moved_in, "d2h_bytes_per_step": moved_out,
           "outputs": list(BatchedUKF.OUTPUT_SETS[cfg["e2e_outputs"]]), "output_set": cfg["e2e_outputs"], "passes_ms": e2e_ms,
           "api": "BatchedUKF.run_host_pipelined, one call per model tile (pinned host inputs -> device -> kernels -> pinned host outputs)"}
    if rank == 0:
        line = base_line(args, cfg, value, world, total_ms / max(len(conc), 1), None)
        line["data"] = "the reference's ship data (fixtures generated from data/historical_ships and data/modern_ships by the unmodified reference)"
        line["config"].update(ships=cfg["job_tracks"], track_steps=steps_all,
                              timed="a 'step' is the whole fleet: each model tile's forward + backward launches on its own stream, CUDA events "
                                    "around the step on the launching stream; L2 flushed between steps; roofline.forward_ms / backward_ms come from a "
                                    "second pass with one launch after the other",
                              ms_per_step_one_stream=(f_ms + b_ms) / max(len(recs), 1))
        line["roofline"] = roofline_block(cfg, steps_local * len(recs), f_ms, b_ms, fp64_probe(lib, nat, torch, dev), args.full_cov)
        line["roofline"]["forward_ms"], line["roofline"]["backward_ms"] = f_ms / len(recs), b_ms / len(recs)
        line["roofline"]["note"] = ("72 tracks occupy one warp on each of three SMs: the step is bound by the latency of one track's sequential "
                                    "time loop (~5 us per filter step), not by HBM or the FP64 pipe")
        line["e2e"], line["gpu_launches"], line["clocks"] = e2e, 2 * len(tiles) * len(conc), clocks.summary()
        line["parity_vs_reference"] = {"worst_smoothed_mean_error": worst, "note": "against the reference's outputs stored in the fixtures"}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"], _ = cpu_baseline_block(args, args.config)
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", default="c5", choices=sorted(CONFIGS))
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tracks", type=int, default=8 * GRANULE, help="tracks per resident tile per GPU (uniform configs)")
    ap.add_argument("--e2e-tracks", type=int, default=GRANULE, help="tracks of the host-buffer end-to-end tile")
    ap.add_argument("--e2e-headline-only", action="store_true", help="time only the config's own output set end to end")
    ap.add_argument("--state-budget", type=float, default=4.0e8, help="stored states per ragged tile (config c4)")
    ap.add_argument("--full-job", action="store_true", help="c4: run every tile of this rank's share, not a stratified K-tile subset")
    ap.add_argument("--no-job", action="store_true", help="c3/c5: skip the whole-job pass")
    ap.add_argument("--no-partitioned", action="store_true", help="c5: skip the SM-partitioned (green context) schedule")
    ap.add_argument("--smoother-sms", type=int, default=48, help="SMs of the smoother's partition in the partitioned schedule")
    ap.add_argument("--in-place", action="store_true", help="smooth in place (halves the state memory)")
    ap.add_argument("--full-cov", action="store_true", help="store full 4x4 covariances (default: the 10 unique entries)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-tracks-per-core", type=int, default=16)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<name>.npy (float64; a fixed, "
                                                          f"seeded sample of track columns, at most {DUMP_BYTES // 10**6} MB)")
    args = ap.parse_args()
    args.state_budget = int(args.state_budget)
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU path computed (--impl b200)")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    args.warmup = max(args.warmup, 3)  # timing rule: at least three warm-up steps
    D = Dist(args)
    try:
        cfg = CONFIGS[args.config]
        (run_fleet if cfg.get("fleet") else run_ragged if cfg["ragged"] else run_uniform)(args, D)
    finally:
        D.close()


if __name__ == "__main__":
    main()
