#!/usr/bin/env python3
"""bench.py — particle-steps/s of the FastSLAM 1.0 hot path.

    python bench.py --gpus N --steps K --warmup W            # our arm (one JSON line on rank 0)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path (oracle port) on the host cores
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR # also write the last timed step's outputs to DIR/*.npy

Primary line (`value`, `e2e`, `roofline`): BASELINE.json config 3 — 65 536 particles x 256 landmarks PER GPU (weak scaling:
global = 65 536 x N), ~12.7 of 256 landmarks observed per step, nth = particles / 1.5.  A "step" = one fastslam_update
(fs1.rs:237-266) over all particles.  Timing: CUDA events on the engine's own stream around every step, L2 flushed (256 MiB
memset + 256 MiB clean read) before each step so no step runs out of a warm cache; `value` = particles x K / sum of step
times (max over ranks).  Inputs (particle state, maps) are resident in HBM; the per-step control + observation list (~300 B)
rides in the launch parameters.  `e2e` repeats K steps through the public API with host buffers, one host synchronisation
and a host read-back of the step's result record (best particle, gate, N_eff) every step.
Second key `c4_strong`: BASELINE config 4 — 2^20 particles x 1024 landmarks sharded over the N GPUs (strong scaling; at
N = 1 the whole 103 GB of landmark state lives on the one GPU), same timing rules, fewer steps.  `--config c4` makes it the
primary line instead.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

# stdout carries exactly one JSON line: whatever NCCL wants to say (its version banner when NCCL_DEBUG is set) goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PARTICLES = 1 << 16          # per GPU (weak scaling: global = N_PARTICLES * n_gpus)
SIDE = 16                      # 16 x 16 = 256 landmarks
BYTES_POSE_WEIGHT = 64         # SURVEY.md §8(d): pose R24+W24, weight R8+W8
BYTES_PER_OBS = 96             # landmark R48+W48 per (particle, observed landmark)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled in the background during the measurement."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                       "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1]))
            except ValueError:
                continue
            for nm, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            busy = [s for s in sm if s >= 0.5 * max(sm)] or sm
            out.update(sm_mhz=statistics.median(busy), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def make_scenario(total_steps):
    from rust_robotics_b200 import scenarios
    return scenarios.c3_scenario(steps=total_steps)


def obs_arrays(rr, sc):
    return [rr.FastSlam1._obs(z) for z in sc.obs]


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's algorithm (oracle port, glibc libm like the Rust reference), all host threads
# ------------------------------------------------------------------------------------------------
VARIANT = 1                # --variant: 1 = fastslam1::fastslam_update (the headline), 2 = fastslam2::fastslam2_update (SURVEY.md 8(f) row 1)
NTH_MODE = "default"       # --nth: default = particles/1.5 (BASELINE config 3 as surveyed), literal = fs1.rs:21's 66.67, every = resample every step


def nth_value(n):
    return {"default": n / 1.5, "literal": 100.0 / 1.5, "every": float(n) + 1.0}[NTH_MODE]


def cpu_run(sc, n, steps, warmup, threads, t0_step=0):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import _oracle
    L = _oracle.load(libm=True)
    o = _oracle.OracleFS(L, n, sc.m, seed=42, variant=VARIANT, nth=nth_value(n))
    L.orc_fs_set_threads(o.h, threads)
    o.seed_map(sc.start, sc.landmarks)
    arrs = [o.obs_array(z) for z in sc.obs]
    import numpy as np
    u = np.asarray(sc.control, dtype=np.float64)
    up = u.ctypes.data_as(_oracle.c_dp)
    for t in range(warmup):
        L.orc_fs_step(o.h, up, arrs[t0_step + t], len(sc.obs[t0_step + t]))
    t0 = time.perf_counter()
    res = 0
    for t in range(warmup, warmup + steps):
        res += L.orc_fs_step(o.h, up, arrs[t0_step + t], len(sc.obs[t0_step + t]))
    dt = time.perf_counter() - t0
    return dt, res


def pick_threads(sc, n):
    """the thread count that serves the CPU arm best on this box (all logical CPUs is often NOT it: shared hosts,
    cgroup quotas, tiny per-thread work); probed with 3-step runs.  Returns (best, seconds per step, {threads: steps/s})."""
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    cands = sorted({c for c in (1, 4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    best, best_dt, table = 1, None, {}
    for c in cands:
        dt, _ = cpu_run(sc, n, 3, 1, c)
        table[c] = round(n * 3 / dt, 1)
        if best_dt is None or dt < best_dt:
            best, best_dt = c, dt
    return best, best_dt / 3, table


def cpu_baseline(sc, budget_s, max_steps):
    """bounded sample of the same workload: same map, same observation stream, fewer particles / steps.  Reported both the
    way the reference runs (ONE thread: the Rust loops are serial) and with the thread count that serves this box best."""
    n = 32768
    threads, per_step, table = pick_threads(sc, n)
    steps = int(max(4, min(max_steps, len(sc.obs) - 4, budget_s / max(per_step, 1e-6))))
    dt, res = cpu_run(sc, n, steps, 2, threads)
    n1 = 4096
    steps1 = int(max(3, min(40, len(sc.obs) - 4)))
    dt1, _ = cpu_run(sc, n1, steps1, 1, 1)
    return {"value": n * steps / dt, "unit": "particle-steps/s", "cores": threads, "kind": "port",
            "one_thread": {"value": n1 * steps1 / dt1, "unit": "particle-steps/s", "sample": f"{n1} particles, {steps1} steps, {dt1:.1f} s"},
            "threads_probe_particle_steps_per_s": table,
            "sample": f"oracle port (C, glibc libm, OpenMP x{threads}) of fs1.rs on {n} of {N_PARTICLES} particles x {sc.m} landmarks, "
                      f"{steps} steps of the same observation stream, {res} resamples, {dt:.1f} s"}


def run_reference(args, rank):
    if rank != 0:
        return
    sc = make_scenario(args.warmup + args.steps + 8)
    # size the per-step sample so the whole run stays within ~2 minutes
    n = 2048
    threads, per_step, _ = pick_threads(sc, n)
    per_ps = per_step / n
    budget = 90.0
    n_fit = budget / (per_ps * (args.steps + args.warmup))
    n = 256
    while n * 2 <= min(n_fit, N_PARTICLES):
        n *= 2
    dt, res = cpu_run(sc, n, args.steps, args.warmup, threads)
    value = n * args.steps / dt
    line = {"impl": "reference", "metric": "particle-steps/sec", "value": value, "unit": "particle-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(CONFIGS["c3"], sc, args.gpus, N_PARTICLES * args.gpus, sc.obs[args.warmup:args.warmup + args.steps], res, args.steps),
            "cpu_baseline": {"value": value, "unit": "particle-steps/s", "cores": threads, "kind": "port",
                             "sample": f"oracle port of fs1.rs (C, glibc libm, OpenMP x{threads}); each step = {n} of "
                                       f"{N_PARTICLES} particles x {sc.m} landmarks, {res} resamples in {args.steps} steps"},
            "e2e": {"value": value, "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def load_traffic():
    """DRAM bytes of one launch of the dominant kernel from the committed `ncu --set full` capture (profiles/*_traffic.json,
    newest round last); null when no capture is committed."""
    import glob
    files = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "*_traffic.json")))
    if not files:
        return {"traffic": None}
    try:
        with open(files[-1]) as f:
            t = json.load(f)
        return {"traffic": t["dram_bytes_read"] + t["dram_bytes_write"], "traffic_source": f"{os.path.basename(files[-1])}: {t['kernel']}"}
    except Exception:
        return {"traffic": None}


# ------------------------------------------------------------------------------------------------
# --dump-outputs: what the timed path computed in its last timed step, as float64 .npy files, so that two builds can be
# compared output for output on identical (seeded) inputs
# ------------------------------------------------------------------------------------------------
DUMP_LIMIT_BYTES = 64 << 20
DUMP_MAP_PARTICLES = 256       # landmark maps are n x m x 48 bytes: a fixed, seeded sample of particles is written
DUMP_ROWS_BYTES = 48 << 20     # larger particle arrays are written as a fixed, seeded sample of rows


def seeded_sample(n, k):
    import numpy as np
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(12345).choice(n, size=k, replace=False))


def sample_rows(name, a, out):
    """a whole when it fits DUMP_ROWS_BYTES, else a fixed, seeded sample of its rows (and `<name>_index`, the rows taken)"""
    per_row = a.nbytes // max(a.shape[0], 1)
    idx = seeded_sample(a.shape[0], max(1, DUMP_ROWS_BYTES // max(per_row, 1)))
    if idx.size == a.shape[0]:
        out[name] = a
    else:
        out[name] = a[idx]
        out[name + "_index"] = idx


def fastslam_outputs(g):
    """what a caller of fastslam_update holds after the step: every particle's (weight, x, y, yaw), the landmark maps
    (x, y, c00, c01, c10, c11 per landmark) of a seeded sample of particles, get_best_particle(), and whether it resampled"""
    import numpy as np
    out = {}
    poses, _ = g.state(landmarks=False)
    sample_rows("particles", poses, out)
    pick = seeded_sample(g.n_local, DUMP_MAP_PARTICLES)
    out["landmarks"] = np.stack([g.particle_landmarks(int(i)) for i in pick])
    out["landmarks_index"] = pick
    best, best_pose = g.get_best_particle()
    out["best_index"] = np.array([best])
    out["best_particle"] = best_pose
    out["resampled"] = np.array([g.last_gate()])
    return out


def pf_outputs(g):
    """what a caller of try_step holds after the step: the particles (x, y, yaw, v, weight) and estimate()"""
    out = {}
    sample_rows("particles", g.get_particles(), out)
    out["estimate"] = g.estimate()
    return out


def write_outputs(d, arrays, suffix=""):
    import numpy as np
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(d, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(d, f"{k}{suffix}.npy"), a)


CONFIGS = {   # SURVEY.md §8(d)
    "c3": dict(name="FastSLAM 1.0 (fs1.rs fastslam_update), BASELINE config 3", particles_per_gpu=N_PARTICLES, particles_total=None,
               scenario="c3_scenario", scaling="weak"),
    "c4": dict(name="FastSLAM 1.0 (fs1.rs fastslam_update), BASELINE config 4", particles_per_gpu=None, particles_total=1 << 20,
               scenario="c4_scenario", scaling="strong"),
}


def workload_config(cfg, sc, n_gpus, n_global, obs_timed, resamples, K):
    return {"workload": cfg["name"] + ("" if VARIANT == 1 else " [FastSLAM 2.0 step, fastslam2.rs]"), "particles": n_global, "particles_per_gpu": n_global // n_gpus, "landmarks": sc.m,
            "mean_obs_per_step": round(sum(len(z) for z in obs_timed) / max(len(obs_timed), 1), 2),
            "resample_fraction": round(resamples / max(K, 1), 3),
            "nth": {"default": "particles/1.5", "literal": "66.67 (fs1.rs:21; never resamples at this particle count)",
                    "every": "particles + 1 (stress variant: resample every step)"}[NTH_MODE],
            "start": "initialised map (cov 10 I), poses at truth", "seed": 42,
            "parallelism": f"particle shards x{n_gpus}" + ("" if n_gpus == 1 else ", peer memory (NVLink loads / stores inside the kernels; no NCCL call, no host sync per step)"),
            "l2": "flushed (256 MiB memset + clean read) before every timed step"}


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def make_engine(rr, grp, cfg_key, rank, world, local_rank):
    from rust_robotics_b200 import dist as rdist, scenarios
    cfg = CONFIGS[cfg_key]
    n_global = cfg["particles_total"] or cfg["particles_per_gpu"] * world
    return cfg, n_global, scenarios, rdist


def measure(rr, grp, cfg_key, K, W, rank, world, local_rank, with_e2e, sampler_cb=None, dump_dir=None):
    """one configuration: warm-up, K flushed + event-timed steps, K un-flushed steps, (optionally) K end-to-end steps.
    dump_dir: write the outputs of the last of the K steps `value` is quoted on (each rank its own shard)"""
    from rust_robotics_b200 import dist as rdist, scenarios
    cfg = CONFIGS[cfg_key]
    n_global = cfg["particles_total"] or cfg["particles_per_gpu"] * world
    total = W + 4 * K + 4
    sc = getattr(scenarios, cfg["scenario"])(steps=total)
    if os.environ.get("BENCH_EMPTY_OBS"):      # experiment: no observations (the EKF launch degenerates to predict; what does the post kernel cost then?)
        sc.obs = [[] for _ in sc.obs]
    arrs = obs_arrays(rr, sc)
    fcfg = rr.FsConfig(nth=nth_value(n_global))
    if world > 1:
        uid = rdist.broadcast_unique_id(grp, rdist.nccl_unique_id)
        g = (rr.FastSlam2 if VARIANT == 2 else rr.FastSlam1)(n_global, sc.m, fcfg, seed=42, device=local_rank, shard=(uid, rank, world))
    else:
        g = (rr.FastSlam2 if VARIANT == 2 else rr.FastSlam1)(n_global, sc.m, fcfg, seed=42, device=local_rank)
    g.seed_map(sc.start, sc.landmarks)

    def barrier():
        g.sync()
        grp.barrier()

    step = 0
    for _ in range(W):                                   # warm-up (untimed)
        g.fastslam_update(sc.control, sc.obs[step], want_flag=False, obs_array=arrs[step]); step += 1
    barrier()
    # ---- timed region 1: K steps, L2 flushed before each, one event pair per step ----
    flush_mode = os.environ.get("BENCH_FLUSH_MODE", "flush")

    def flushed_pass(kernel_events):
        nonlocal step
        s0 = g.stats()
        g.time_main_kernel(kernel_events)
        barrier()
        first = step
        for t in range(K):
            if flush_mode != "none":
                g.flush_l2()
            g.mark(2 * t)
            g.fastslam_update(sc.control, sc.obs[step], want_flag=False, obs_array=arrs[step]); step += 1
            g.mark(2 * t + 1)
        barrier()
        ms = [g.elapsed_ms(2 * t, 2 * t + 1) for t in range(K)]
        s1 = g.stats()
        g.time_main_kernel(False)
        return first, ms, s0, s1

    # pass A: the K steps `value` is quoted on.  No events inside a step: an event pair around the EKF launch costs ~8 us per step (it
    # breaks the programmatic dependent launch of the kernel behind it), so the kernel is timed on its own pass below.
    first, step_ms, st0, st1 = flushed_pass(False)
    if dump_dir:
        write_outputs(dump_dir, fastslam_outputs(g), "" if world == 1 else f"_rank{rank}")
    if os.environ.get("BENCH_VERBOSE") and rank == 0:
        ss = sorted(step_ms)
        sys.stderr.write("step ms: min %.3f  p50 %.3f  p90 %.3f  p99 %.3f  max %.3f  sum %.1f; worst steps %s\n" % (
            ss[0], ss[len(ss) // 2], ss[int(len(ss) * 0.9)], ss[int(len(ss) * 0.99)], ss[-1], sum(ss),
            sorted(range(K), key=lambda i: -step_ms[i])[:8]))
    t_flushed = grp.max(sum(step_ms) * 1e-3)
    launches = st1.kernel_launches - st0.kernel_launches
    resamples = st1.resamples - st0.resamples
    obs_timed = sc.obs[first:first + K]
    n_local = n_global // world
    # pass B: the next K steps, same protocol, with a CUDA event pair around every launch of the dominant kernel (roofline)
    first_b, step_ms_b, _, stb = flushed_pass(True)
    kernel_ms = stb.main_kernel_ms_sum / max(stb.main_kernel_count, 1)
    alg_bytes = sum(n_local * (BYTES_POSE_WEIGHT + BYTES_PER_OBS * len(z)) for z in sc.obs[first_b:first_b + K]) / K
    t_flushed_b = grp.max(sum(step_ms_b) * 1e-3)
    # ---- timed region 2: the next K steps back to back, no flush (steady state, informational) ----
    barrier()
    g.mark(8000)
    for t in range(K):
        g.fastslam_update(sc.control, sc.obs[step], want_flag=False, obs_array=arrs[step]); step += 1
    g.mark(8001)
    barrier()
    t_noflush = grp.max(g.elapsed_ms(8000, 8001) * 1e-3)
    # ---- end to end: public API, host buffers in, the step's result record read back to the host every step ----
    e2e = None
    if with_e2e:
        barrier()
        t0 = time.perf_counter()
        h2d = d2h = 0
        # One step in flight at a time.  The host builds step t+1's C observation array from host data while the device runs
        # step t (ordinary double buffering on the caller's side), then synchronises on step t and reads its result record.
        arr_next = g._obs(sc.obs[step])
        for t in range(K):
            z, arr = sc.obs[step], arr_next
            g.fastslam_update(sc.control, z, want_flag=False, obs_array=arr); step += 1   # enqueue: control + observations ride in the launch parameters
            if t + 1 < K:
                arr_next = g._obs(sc.obs[step])
            idx, pose = g.get_best_particle()                                          # synchronises; the 64-byte record: best particle + pose, gate, N_eff
            h2d += 16 + 24 * len(z)
            d2h += 64
        barrier()
        t_e2e = grp.max(time.perf_counter() - t0)
        e2e = {"value": n_global * K / t_e2e, "unit": "particle-steps/s", "h2d_bytes_per_step": h2d / K, "d2h_bytes_per_step": d2h / K,
               "l2": "not flushed: the steps run back to back through the API, one in flight at a time (compare value_steady_state_no_flush)"}
    if rank == 0 and os.environ.get("PFGPU_POST_TRACE"):
        import ctypes as C
        out = (C.c_ulonglong * 32)()
        g.L.pfgpu_fs_post_trace(g.h, out)
        nl = max(out[31], 1)
        nr = max(int(g.stats().resamples), 1)
        us = lambda k, den: out[k] / den / 1e3
        sys.stderr.write("fs3_post_kernel (us, CTA 0; per launch): load+offsets=%.2f  S sum=%.2f [classify+publish %.2f | barrier %.2f | chain %.2f]  "
                         "normalise+gate=%.2f   launches=%d\n" % (us(0, nl), us(1, nl), us(8, nl) + us(28, nl) + us(29, nl) + us(30, nl), us(9, nl), us(10, nl), us(2, nl), nl))
        sys.stderr.write("   per RESAMPLE (%d): S2 sum=%.2f  CDF scan=%.2f [classify+publish %.2f | barrier %.2f | chain %.2f | emit %.2f]  comb+barrier=%.2f  "
                         "search+clone=%.2f\n" % (nr, us(3, nr), us(4, nr), us(12, nr), us(13, nr), us(14, nr), us(15, nr), us(5, nr), us(6, nr)))
        sys.stderr.write("   S classify split: first pass=%.2f  scan=%.2f  classify pass=%.2f  scan+publish=%.2f\n" % (us(28, nl), us(29, nl), us(30, nl), us(8, nl)))
        sys.stderr.write("   step timeline (us per step; globaltimer, CTA 0 / last warp out): idle before the EKF launch=%.2f  EKF launch=%.2f  idle between=%.2f  "
                         "post launch=%.2f (every CTA through its phases after %.2f, then the last one: best particle, record, flip)\n" % (us(7, nl), us(24, nl), us(25, nl), us(26, nl), us(27, nl)))
        nld = max(out[21], 1)
        sys.stderr.write("   leader chain of S (CTA 0 led %d of %d): loads=%.2f tile prefix=%.2f rank=%.2f walk+cert=%.2f publish=%.2f | clone phase per resample: bracket=%.2f stage=%.2f slots=%.2f\n" %
                         (out[21], nl, us(16, nld), us(17, nld), us(18, nld), us(19, nld), us(20, nld), us(22, nr), us(23, nr), us(6, nr)))
    res = {"cfg": cfg, "sc": sc, "n_global": n_global, "t_flushed": t_flushed, "t_noflush": t_noflush, "launches": int(launches),
           "resamples": int(resamples), "kernel_ms": kernel_ms, "t_flushed_kernel_pass": t_flushed_b, "alg_bytes": alg_bytes, "obs_timed": obs_timed, "e2e": e2e,
           "serial_fallbacks": int(st1.serial_fallbacks), "K": K}
    g.close()
    return res


def run_ours(args, rank, world, local_rank):
    import rust_robotics_b200 as rr
    from rust_robotics_b200 import dist as rdist
    grp = rdist.TcpGroup()
    K, W = args.steps, args.warmup
    sampler = ClockSampler(local_rank) if rank == 0 else None
    primary = measure(rr, grp, args.config, K, W, rank, world, local_rank, True, dump_dir=args.dump_outputs)
    second_key = "c4" if args.config == "c3" else "c3"
    second = None
    if not args.no_second:
        K2 = min(K, 50 if second_key == "c4" else K)
        second = measure(rr, grp, second_key, K2, max(3, min(W, 5 if second_key == "c4" else W)), rank, world, local_rank, False)
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        peak, peak_src = load_peaks()
        r = primary
        achieved = r["alg_bytes"] / (r["kernel_ms"] * 1e-3) / 1e9
        cpu = cpu_baseline(r["sc"], 12.0, 400) if (world == 1 and not args.no_cpu_baseline and args.config == "c3") else None
        line = {"metric": "particle-steps/sec", "value": r["n_global"] * K / r["t_flushed"], "unit": "particle-steps/s",
                "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": r["t_flushed"] / K * 1e3, "higher_is_better": True,
                "scaling": r["cfg"]["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": workload_config(r["cfg"], r["sc"], world, r["n_global"], r["obs_timed"], r["resamples"], K),
                "value_steady_state_no_flush": r["n_global"] * K / r["t_noflush"],
                "e2e": r["e2e"], "gpu_launches": r["launches"],
                "roofline": {"bound": "hbm", "kernel": "fs3_ekf_kernel (predict + per-observation EKF + weight products, fs1.rs:245-256)",
                             "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, **load_traffic(),
                             "algorithmic_bytes_per_launch": r["alg_bytes"], "avg_launch_ms": r["kernel_ms"],
                             "timed_on": "a second pass of K flushed steps with a CUDA event pair around every launch of this kernel; those steps took "
                                         "%.4f ms each (the event pairs break the programmatic dependent launch), so `value` is quoted on the pass without them"
                                         % (r["t_flushed_kernel_pass"] / K * 1e3),
                             "note": "per GPU; algorithmic bytes = particles x (64 + 96 x observations of the step), SURVEY.md 8(d)"},
                "clocks": clocks, "serial_fallbacks": r["serial_fallbacks"]}
        if second:
            q = second
            line[{"c4": "c4_strong", "c3": "c3_weak"}[second_key]] = {
                "value": q["n_global"] * q["K"] / q["t_flushed"], "unit": "particle-steps/s", "steps": q["K"], "ms_per_step": q["t_flushed"] / q["K"] * 1e3,
                "scaling": q["cfg"]["scaling"], "value_steady_state_no_flush": q["n_global"] * q["K"] / q["t_noflush"],
                "ekf_launch_ms": q["kernel_ms"], "ekf_roofline_frac": q["alg_bytes"] / (q["kernel_ms"] * 1e-3) / 1e9 / peak,
                "config": workload_config(q["cfg"], q["sc"], world, q["n_global"], q["obs_timed"], q["resamples"], q["K"])}
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    grp.barrier()
    grp.close()


# ------------------------------------------------------------------------------------------------
# secondary workloads (BASELINE configs 2 and 5): MonteCarloLocalizer / ParticleFilterLocalizer, single GPU
# ------------------------------------------------------------------------------------------------
def run_pf(args):
    import numpy as np
    import rust_robotics_b200 as rr
    from rust_robotics_b200 import scenarios
    K, W = args.steps, args.warmup
    n = args.particles
    mcl = args.workload == "mcl"
    sc = scenarios.PfScenario("c2" if mcl else "c1", steps=W + 3 * K + 2)
    if mcl:   # C2: min == max == n, 360 range beams, noises of mcl.rs:490-498
        g = rr.MonteCarloLocalizer.try_with_initial_state(sc.init, rr.MonteCarloLocalizationConfig(n, n, 0.05, 2.326, 0.25, 0.05, 0.02, 0.1), seed=42)
    else:     # C5: the C1 model (5 landmarks), resample_threshold from --threshold
        g = rr.ParticleFilterLocalizer.try_with_initial_state(sc.init, rr.ParticleFilterConfig(n, args.threshold, 0.25), seed=42)
    obs = [np.ascontiguousarray(o) for o in sc.obs]
    ctl = [np.asarray(c, dtype=np.float64) for c in sc.controls]
    t = 0
    for _ in range(W):
        g.try_step(ctl[t], obs[t], want_estimate=False); t += 1
    g.sync()
    sampler = ClockSampler(0)
    # pass A (`value`): K flushed steps, one event pair per step, none inside a step (the fused step of a small filter replays
    # a CUDA graph; per-kernel events would force plain launches).  pass B: K more flushed steps with an event pair around every
    # launch of the dominant kernel (roofline).
    def flushed(kernel_events):
        nonlocal t
        s0 = g.stats()
        g.time_main_kernel(kernel_events)
        for k in range(K):
            g.flush_l2()
            g.mark(2 * k)
            g.try_step(ctl[t], obs[t], want_estimate=False); t += 1
            g.mark(2 * k + 1)
        g.sync()
        dt_ = sum(g.elapsed_ms(2 * k, 2 * k + 1) for k in range(K)) * 1e-3
        s1 = g.stats()
        g.time_main_kernel(False)
        return dt_, s0, s1
    tt, st0, st1 = flushed(False)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, pf_outputs(g))
    tt_b, _, stb = flushed(True)
    t0 = time.perf_counter()
    for k in range(K):
        est = g.try_step(ctl[t], obs[t]); t += 1           # host buffers in, estimate read back every step
    g.sync()
    te = time.perf_counter() - t0
    clocks = sampler.stop()
    kobs = obs[0].shape[0]
    kms = stb.main_kernel_ms_sum / max(stb.main_kernel_count, 1)
    peak, peak_src = load_peaks()
    alg = n * 72.0                                           # pose record R32 + W32, raw weight W8
    line = {"metric": "particle-steps/sec", "value": n * K / tt, "unit": "particle-steps/s", "n_gpus": 1, "steps": K, "warmup": W,
            "ms_per_step": tt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": ("MonteCarloLocalizer try_step (mcl.rs:291-300), BASELINE config 2" if mcl else
                                    "ParticleFilterLocalizer try_step (pf.rs:488-497), BASELINE config 5 point"),
                       "particles": n, "observations_per_step": kobs, "resample_threshold": None if mcl else args.threshold,
                       "resamples_in_timed_steps": int(st1.resamples - st0.resamples), "l2": "flushed before every timed step"},
            "e2e": {"value": n * K / te, "unit": "particle-steps/s", "h2d_bytes_per_step": 16 + 24 * kobs, "d2h_bytes_per_step": 32},
            "gpu_launches": int(st1.kernel_launches - st0.kernel_launches),
            "roofline": {"bound": "hbm", "kernel": "pf_predict_weight_kernel (predict + range likelihood, pf.rs:279-329)",
                         "achieved": alg / (kms * 1e-3) / 1e9, "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                         "frac": alg / (kms * 1e-3) / 1e9 / peak, "traffic": None, "algorithmic_bytes_per_launch": alg, "avg_launch_ms": kms,
                         "timed_on": "a second pass of K flushed steps with an event pair around every launch of this kernel (%.4f ms per step)" % (tt_b / K * 1e3),
                         "note": "FP64-bound when observations_per_step is large (config 2: 360 sqrt+exp+div per particle)",
                         # SURVEY.md 8(d): config 2 is bounded by the FP64 pipe, not HBM: the reference's formula costs 12 f64 operations per
                         # (particle, beam) counting sqrt / exp / div as one each (pf.rs:317-328,476-479) + 13 per particle for predict
                         "fp64_algorithmic_tflops": n * (12.0 * kobs + 13.0) / (kms * 1e-3) / 1e12,
                         "fp64_peak_tflops_nominal": 37.2},
            "clocks": clocks, "serial_fallbacks": int(st1.serial_fallbacks)}
    if not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import _oracle
        L = _oracle.load(libm=True)
        nc = min(n, 1 << 16)
        threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        threads = min(threads, 64)
        o = _oracle.OraclePF(L, nc, threshold=args.threshold, range_noise=0.25, velocity_noise=0.05 if mcl else 2.0,
                             yaw_rate_noise=0.02 if mcl else np.deg2rad(40.0), mode=1 if mcl else 0, max_particles=nc)
        L.orc_pf_set_fast_search(o.h, 1); L.orc_pf_set_threads(o.h, threads)
        o.init_state(sc.init)
        t0 = time.perf_counter(); ks = 0
        while ks < K and time.perf_counter() - t0 < 12.0:
            o.step(ctl[ks], obs[ks]); ks += 1
        dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": nc * ks / dt, "unit": "particle-steps/s", "cores": threads, "kind": "port",
                                "sample": f"oracle port of {'mcl.rs' if mcl else 'pf.rs'} (C, glibc libm, OpenMP x{threads} over particles, lower_bound "
                                          f"index search = reference-equivalent), {nc} particles, {ks} steps, {dt:.1f} s"}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU leg (profiling runs)")
    ap.add_argument("--workload", default="fastslam", choices=["fastslam", "mcl", "pf"],
                    help="fastslam = BASELINE config 3 (default, the headline); mcl = config 2; pf = one point of the config-5 sweep")
    ap.add_argument("--config", default="c3", choices=["c3", "c4"], help="fastslam workload: which BASELINE config is the primary line (the other one is reported under a second key)")
    ap.add_argument("--no-second", action="store_true", help="skip the second configuration")
    ap.add_argument("--nth", default="default", choices=["default", "literal", "every"],
                    help="fastslam workload: resample threshold — particles/1.5 (default), the reference's literal 66.67, or every step")
    ap.add_argument("--variant", type=int, default=1, choices=[1, 2],
                    help="fastslam workload: 1 = FastSLAM 1.0 (the headline), 2 = FastSLAM 2.0 (fastslam2.rs) on the same configurations")
    ap.add_argument("--particles", type=int, default=1 << 20, help="mcl / pf workloads only")
    ap.add_argument("--threshold", type=float, default=1.0, help="pf workload: resample_threshold (1.0 = resample every step)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of the K steps `value` is quoted on computed to DIR/<name>.npy "
                         "(float64; large arrays as a fixed, seeded sample; at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference" and args.workload == "fastslam":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    global NTH_MODE, VARIANT
    NTH_MODE = args.nth
    VARIANT = args.variant
    if args.warmup < 3:
        args.warmup = 3
    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.workload != "fastslam":
        if rank == 0:
            run_pf(args)
        return
    if args.impl == "reference":
        run_reference(args, rank)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
