#!/usr/bin/env python
"""bench.py — spin-updates/s of the IsingModel.jl spin-update hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload all|c1|c2|c3|c4|c5]

Default (`--workload all`): ONE JSON line whose top level is the headline — BASELINE.json configs[1], "SK dense
Gaussian J, N=1024, 4096 replicas, Glauber sweeps with annealing schedule" per GPU (weak scaling, replicas sharded,
no data-path collective: SURVEY §8e) — timed over exactly --steps steps after --warmup warm-ups, and whose
`workloads` object carries, measured in the same process, the other BASELINE configs:
  c1  32x32 periodic ferromagnet, Metropolis at T = 2.269, 10^4 sweeps, 4096 replicas + the R = 1 latency
  c3  dense N = 4096 MultiSpinFlip SCA, 8192 replicas     (tcgen05 contraction; primary = exact-split int8 planes)
  c4  bipartite 784 x 512 block Gibbs, 16384 chains        (chain-resident tcgen05 kernel)
  c5  (--gpus N > 1 only) dense N = 8192 x N rows sharded, 1024 replicas, spins exchanged every half-step
Each sub-result has its own `value`, `roofline`, `e2e`, `clocks`, `cpu_baseline` and a timed region of >= 2 s
(`steps` chosen from the warm-up time, the same on every rank).  `--workload cX` prints that workload alone as the line.

  value     : device-timed (CUDA events on the launching stream, per step, max over ranks), inputs resident in
              HBM, noise drawn by the in-kernel Philox RNG.
  e2e       : the same run through the public host API (isingmodel.jl_b200: SpinSystems / SingleSpinFlip /
              OnBipartiteGraph / SamplingHelper.run_), timed on the host with pinned buffers: H2D of the initial spins
              and the schedule, the steps, D2H of the final spins, energies and flip counts.
  roofline  : the dominant kernel against what binds it: the tensor pipe for the contractions (measured cuBLAS bf16
              burst rate), the shared-memory pipe for the dense sweep kernel (J rows are staged once per CTA and read
              by its chains from shared memory: DRAM traffic is 46 MB per launch, the HBM roof is moot and the SURVEY
              §8d flips x N x 8 B figure is kept as an auxiliary field), the issue slots for the lattice kernel.
  cpu_baseline / --impl reference : the CPU oracle (C restatement of the reference's algorithm: a full Float64 row
              dot per update; Julia is not installed here), on all host cores and on 1 thread (the reference itself
              is single-threaded: src/SamplingHelper.jl:42-50).

  --dump-outputs DIR : after the timed steps, what the last timed step of the printed workload computed, as
              DIR/<name>.npy (spins in float32, flip counts in float64), so that two builds can be compared output for
              output: the inputs depend only on the arguments.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from, which may be read-only

import numpy as np  # noqa: E402

N_SITES, REPLICAS = 1024, 4096
T0, TF = 2.0, 0.05
SEED_J, SEED_S = 2, 3
METRIC, UNIT = "spin-updates/sec", "updates/s"
SUB_TIMED_MS = 2200.0          # timed region of every sub-workload (>= 2 s: clocks are sampled every 50 ms)
PREC_PASSES = {"bf16x3": 3.0, "bf16x2": 2.0, "bf16x1": 1.0, "fp16x2": 2.0, "fp16x1": 1.0, "f64": 1.0,
               "i8x3": 1.5, "i8x2": 1.0, "i8x4": 2.0}      # tensor passes in bf16-pass equivalents (int8 runs at 2x)
PREC_NOTE = {"i8x3": "exact split: 24-bit fixed-point couplings as 3 int8 digit planes, exact int32 accumulation",
             "i8x4": "exact split: 32-bit fixed-point couplings as 4 int8 digit planes, exact int32 accumulation",
             "i8x2": "16-bit fixed-point couplings as 2 int8 digit planes, exact int32 accumulation",
             "fp16x2": "exact split: 2 fp16 terms (2^-24 of max|W|), fp32 accumulation",
             "bf16x3": "exact split: 3 bf16 terms (2^-27 of max|W|), fp32 accumulation",
             "bf16x2": "2 bf16 terms (2^-18), fp32 accumulation",
             "bf16x1": "ROUNDED J: couplings rounded to one bf16 term (8 bits) — not the reference's model",
             "fp16x1": "ROUNDED J: couplings rounded to one fp16 term (11 bits) — not the reference's model",
             "f64": "Float64 kernel (no tensor cores)"}


def workload(sweeps):
    from isingmodel_jl_b200 import synth
    J = synth.sk_J(N_SITES, SEED_J)
    h = np.zeros(N_SITES)
    T = synth.geometric_schedule(T0, TF, sweeps)
    return J, h, T


def c2_config(args):
    """The headline's `config`: identical in the GPU arm and in the reference arm (the driver compares them)."""
    return {"workload": "C2: Sherrington-Kirkpatrick dense Gaussian J, N=1024, 4096 replicas/GPU, Glauber "
                        f"sequential sweeps, geometric annealing T {T0}->{TF} over {args.sweeps} sweeps",
            "n_sites": N_SITES, "replicas_per_gpu": REPLICAS, "sweeps_per_step": args.sweeps,
            "updates_per_step_per_gpu": N_SITES * REPLICAS * args.sweeps, "sharding": "replicas (no collective)",
            "l2": "flushed between timed steps (256 MiB write); J (8 MiB) is L2/smem-resident by design"}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        pk = json.load(open(path))
        return {"hbm": float(pk["hbm_gbs"]), "tc_burst": float(pk["bf16_tflops"]),
                "tc_sustained": float(pk.get("bf16_tflops_sustained", pk["bf16_tflops"])), "src": "MEASURED_PEAKS.json (of measured)"}
    return {"hbm": 6650.0, "tc_burst": 1590.0, "tc_sustained": 1400.0, "src": "B200_PROFILING.md fallback (of fallback)"}


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.proc = None

    def window(self, t_lo, t_hi):
        """Summary of the samples taken inside [t_lo, t_hi] (time.time() bounds of a timed region)."""
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        inside = [r for t, r in list(self.rows) if t_lo <= t <= t_hi + 0.05]
        scope = "timed region"
        if len(inside) < 3:  # a very short timed region: every sample under load so far
            inside, scope = [r for _, r in list(self.rows)], "warm-up + timed region"
        for r in inside:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                pw.append(float(r[3]))
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


# ---------------------------------------------------------------------------------------------- runtime (GPU arm)
class Runtime:
    """One process per GPU: torch is plumbing (stream, events, NCCL barrier / max-over-ranks), nothing else."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.nccl_log = None
        if self.world > 1:
            # NCCL's own communicator lines (ranks, transport, NVLS) go to a file and are quoted in the c5 sub-result
            self.nccl_log = os.path.join(tempfile.gettempdir(), f"isb_nccl_{os.getpid()}.log")
            os.environ.setdefault("NCCL_DEBUG", "INFO")
            os.environ.setdefault("NCCL_DEBUG_SUBSYS", "INIT")
            os.environ.setdefault("NCCL_DEBUG_FILE", self.nccl_log)
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
        from isingmodel_jl_b200 import _lib, sharding
        self.L, self.sharding = _lib, sharding
        self.stream = torch.cuda.Stream()
        torch.cuda.set_stream(self.stream)
        self.ctx = _lib.context(self.local)
        self.ctx.set_stream(self.stream.cuda_stream)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        self.sms = int(torch.cuda.get_device_properties(self.local).multi_processor_count)
        self.sampler = ClockSampler(self.local)
        if self.rank == 0:
            self.sampler.start()
        self.last_stats = lambda: {}

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v):
        return self.sharding.max_over_ranks(v)

    def pinned(self, shape):
        return self.torch.empty(shape, dtype=self.torch.int8).pin_memory().numpy()

    def timed(self, fn):
        """fn() enqueues one step on self.stream; returns its device time in ms (CUDA events on that stream)."""
        torch = self.torch
        self.flush.zero_()                                   # L2 flush (256 MiB > 126 MB)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        fn()
        e1.record(self.stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def run_steps(self, reset, step, warmup, steps):
        """`warmup` untimed then exactly `steps` timed steps (steps=None: as many as fill SUB_TIMED_MS, decided from the
        last warm-up's time, max over ranks, so every rank runs the same count); barrier + synchronize on both sides.
        Returns (steps, device seconds summed over the timed steps and maxed over ranks, per-step stats, clocks)."""
        last = 0.0
        for k in range(warmup):
            reset()
            last = self.timed(lambda: step(k))
        if steps is None:
            t_w = self.max_over_ranks(last)
            steps = int(min(400, max(3, math.ceil(SUB_TIMED_MS / max(t_w, 1e-3)))))
        self.barrier()
        t_lo = time.time()
        ms, stats = [], []
        for k in range(steps):
            reset()
            ms.append(self.timed(lambda: step(warmup + k)))
            stats.append(self.last_stats())
        self.barrier()
        t_hi = time.time()
        clocks = self.sampler.window(t_lo, t_hi) if self.rank == 0 else None
        return steps, self.max_over_ranks(sum(ms) / 1e3), stats, clocks

    def close(self):
        self.sampler.stop()
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def captured_traffic(key):
    """DRAM bytes per launch of a dominant kernel from its committed `ncu --set full` capture (profiles/roofline_traffic.json)."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "roofline_traffic.json")))["other_kernels"][key]
        return float(d["bytes"]), d["source"]
    except Exception:
        return None, None


def tensor_peak(pk, t_dev):
    """The tensor-roofline denominator for a timed region of `t_dev` device seconds, as MEASURED_PEAKS.json defines its two
    figures: the cuBLAS bf16 BURST rate for a kernel timed alone in a short region, the SUSTAINED rate (cuBLAS back to back
    for 4 s: the chip power-caps to ~1.3 GHz) for a kernel timed inside a long step.  Regions of 2 s and more count as long;
    both fractions are always reported beside `frac`."""
    if t_dev >= 2.0:
        return pk["tc_sustained"], (f"{pk['src']}: cuBLAS bf16 SUSTAINED rate — the timed region is {t_dev:.1f} s of back-to-back "
                                    "launches (power-capped clocks, see `clocks`); `frac_of_burst` is given beside it")
    return pk["tc_burst"], (f"{pk['src']}: cuBLAS bf16 BURST rate — the timed region is only {t_dev:.2f} s; "
                            "`frac_of_sustained` is given beside it")


def base_line(value, world, steps, warmup, ms_per_step, dtype, cfg):
    return {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": dtype, "data": "synthetic", "config": cfg}


DUMP_BYTES = 60 << 20          # below 64 MB (decimal) with the .npy headers


def dump_outputs(path, arrays):
    """--dump-outputs: `arrays` (name -> one row per replica) as path/<name>.npy, int8 spins as float32 and everything
    else as float64.  Above DUMP_BYTES in all, every array keeps the same fixed, seeded sample of replicas (sorted)."""
    os.makedirs(path, exist_ok=True)
    out = {k: np.asarray(a, dtype=np.float32 if np.asarray(a).dtype == np.int8 else np.float64) for k, a in arrays.items()}
    R = len(next(iter(out.values())))
    row_bytes = sum(a[0].nbytes for a in out.values())
    keep = slice(None)
    if R * row_bytes > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(R, DUMP_BYTES // row_bytes, replace=False))
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), a[keep])


# ---------------------------------------------------------------------------------------------- CPU arm (oracle)
def c2_cpu_rate(sweeps_total, seconds_target, threads=None):
    """Times the CPU oracle (one chain per thread, full Float64 row dot per update) on a bounded sample of the C2
    workload; returns (updates/s, description, threads)."""
    import oracle
    from isingmodel_jl_b200 import synth
    threads = threads or oracle.num_threads()
    J, h, T = workload(sweeps_total)
    R = threads
    S0 = synth.spins(SEED_S, R, N_SITES)

    def run(nsw):
        nsteps = nsw * N_SITES
        fl = synth.logistic(5, (R, nsteps))
        t0 = time.perf_counter()
        oracle.ssf_run_batch(oracle.GLAUBER, J, h, S0, nsteps, fluct=fl, fluct_per_replica=True, T=T[:nsw],
                             steps_per_T=N_SITES, nthreads=threads)
        return time.perf_counter() - t0, nsteps * R

    dt, n = run(2)  # calibration (also warms the caches)
    nsw = int(max(2, min(sweeps_total, round(2 * seconds_target / max(dt, 1e-6)))))
    reps = int(max(1, round(seconds_target / max(dt * nsw / 2, 1e-6))))
    dt, n = 0.0, 0
    for _ in range(reps):
        d, m = run(nsw)
        dt, n = dt + d, n + m
    return n / dt, (f"{R} chain(s) (one per thread) x first {nsw} sweeps of the C2 schedule x {reps} repeats "
                    f"({n} updates, {dt:.1f} s wall)"), threads


def c1_cpu_rate(seconds, threads=None):
    import oracle
    from isingmodel_jl_b200 import synth
    threads = threads or oracle.num_threads()
    N, T1 = 1024, 2.269
    J = synth.lattice_J(32)
    S0 = synth.spins(SEED_S, threads, N)

    def run(nsw):
        fl = synth.exponential(5, (threads, nsw * N))
        t0 = time.perf_counter()
        oracle.ssf_run_batch(oracle.METROPOLIS, J, np.zeros(N), S0, nsw * N, fluct=fl, fluct_per_replica=True,
                             T=np.array([T1]), steps_per_T=nsw * N, nthreads=threads)
        return time.perf_counter() - t0

    dt = run(4)  # calibration
    nsw = int(max(4, min(4000, round(4 * seconds / max(dt, 1e-6)))))
    dt = run(nsw)
    return threads * nsw * N / dt, (f"{threads} chain(s) (one per thread) x {nsw} sweeps ({dt:.1f} s wall), dense-row dot "
                                    "per update as the reference does"), threads


def sca_cpu_rate(W, h, b, T, seconds_target, threads=None):
    """Times the CPU oracle's SCA (two Float64 mat-vecs per step and chain, src/OnBipartiteGraph.jl:35-42) on a bounded sample
    of about `seconds_target` wall seconds: first more steps (up to 200), then more chains per thread."""
    import oracle
    from isingmodel_jl_b200 import synth
    threads = threads or oracle.num_threads()
    nv, nh = W.shape

    def run(n, per_thread):
        R = threads * per_thread
        S0, H0 = synth.spins(7, R, nv), synth.spins(8, R, nh)
        Fv, Fh = synth.logistic(9, (n, nv), 1), synth.logistic(9, (n, nh), 2)
        t0 = time.perf_counter()
        oracle.bip_run_batch(oracle.SCA, W, h, b, S0, H0, n, Fv, Fh, T[:n] if len(T) >= n else np.resize(T, n), nthreads=threads)
        return time.perf_counter() - t0, n * (nv + nh) * R

    run(1, 1)                                  # (first call: library load, page faults)
    dt, cnt = run(2, 1)
    dt /= 2.0
    n = int(max(1, min(200, round(seconds_target / max(dt, 1e-6)))))
    per_thread = int(max(1, min(256, round(seconds_target / max(dt * n, 1e-6)))))
    dt, cnt = run(n, per_thread)
    return cnt / dt, f"{threads * per_thread} chain(s) ({per_thread} per thread, {threads} thread(s)) x {n} SCA steps ({cnt} updates, {dt:.1f} s wall)", threads


def cpu_baselines(fn, seconds):
    """All host cores and one thread (the reference is single-threaded) for the same kind of bounded sample."""
    v, sd, cores = fn(seconds, None)
    v1, sd1, _ = fn(max(3.0, seconds / 3.0), 1)
    return {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sd,
            "one_thread": {"value": v1, "unit": UNIT, "cores": 1, "sample": sd1}}


def reference_arm(args, out):
    """--impl reference: the reference's CPU algorithm (oracle port; Julia is not installed) on all host cores, on the
    headline's config, each step a bounded sample of the workload."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0
    which = "c2" if args.workload == "all" else args.workload
    if which == "c5":
        out.write(json.dumps({"impl": "reference", "unavailable": "config 5 (N=65536: J is 32 GiB in Float64) is GPU-only; see --workload c3 for the CPU arm of the same algorithm"}) + "\n")
        out.flush()
        return 0
    if which in ("c3", "c4"):
        W, h, b, R, sched, desc0 = sca_workload(which)
        nst = args.sca_steps or SCA_STEPS[which]
        Tsch = sched(nst)
        fn = lambda s, t=None: sca_cpu_rate(W, h, b, Tsch, s, t)  # noqa: E731
        cfg, upd = sca_config(which, desc0, W, R, nst), (W.shape[0] + W.shape[1]) * R * nst
    elif which == "c1":
        fn = lambda s, t=None: c1_cpu_rate(s, t)  # noqa: E731
        cfg, upd = c1_config(args), 1024 * 4096 * args.c1_sweeps
    else:
        fn = lambda s, t=None: c2_cpu_rate(args.sweeps, s, t)  # noqa: E731
        cfg, upd = c2_config(args), N_SITES * REPLICAS * args.sweeps
    rates, desc, threads = [], "", 1
    for i in range(args.warmup + args.steps):
        rate, desc, threads = fn(args.ref_seconds)
        if i >= args.warmup:
            rates.append(rate)
    v = float(np.mean(rates))
    line = base_line(v, args.gpus, args.steps, args.warmup, 1e3 * upd / v, "f64", cfg)
    line.update({"impl": "reference",
                 "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
                 "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                 "gpu_launches": 0,
                 "note": "CPU restatement of the reference algorithm (Julia unavailable); ms_per_step extrapolated from "
                         "the bounded sample of each step"})
    out.write(json.dumps(line) + "\n")
    out.flush()
    return 0


# ---------------------------------------------------------------------------------------------- C2: dense sweeps
def run_c2(rt, args, steps, warmup, cpu=True, dump=None):
    from isingmodel_jl_b200 import synth, SpinSystems, SingleSpinFlip, SamplingHelper
    L = rt.L
    sweeps = args.sweeps
    nsteps = sweeps * N_SITES
    J, h, T = workload(sweeps)
    prec_name = args.prec if args.prec in ("f64", "f32") else "f64"
    prec = L.PREC_F64 if prec_name == "f64" else L.PREC_F32
    bJ = 8 if prec_name == "f64" else 4
    # this rank's replicas: global replica ids [rank*R, (rank+1)*R) -> distinct initial spins and noise streams
    S0p = rt.pinned((REPLICAS, N_SITES))
    S0p[:] = synth.spins(SEED_S + 1000 * rt.rank, REPLICAS, N_SITES)
    ss = SpinSystems.SpinSystem(S0p, J, h, device=rt.local, prec=prec)
    ua = SingleSpinFlip.GlauberDynamics(ss, T0)
    ens = ss._ensemble()
    rt.last_stats = ens.last_stats
    last = {}

    def step(k):
        last["out"] = ens.ssf_run(L.RULE_GLAUBER, nsteps, order=L.ORDER_SEQUENTIAL, seed=12345 + rt.rank,
                                  step_offset=k * nsteps, T=T, steps_per_T=N_SITES)

    steps, t_dev, stats, clocks = rt.run_steps(lambda: ens.set_spins(S0p), step, warmup, steps)
    if dump and rt.rank == 0:
        dump_outputs(dump, {"spins": ens.get_spins(), "flips": last["out"]["flips"]})

    def e2e_step(k):
        rt.flush.zero_()
        rt.torch.cuda.synchronize()
        t0 = time.perf_counter()
        ss.spinConfiguration = S0p              # H2D (pinned)
        SamplingHelper.run_(ua, nsteps, order="sequential", seed=12345 + rt.rank, step_offset=k * nsteps,
                            temperatures=T, steps_per_T=N_SITES)
        st = ens.last_stats()
        S = ss.spinConfiguration                # D2H
        E = SpinSystems.calcEnergy(ua)          # D2H
        rt.torch.cuda.synchronize()
        return time.perf_counter() - t0, S0p.nbytes + st["h2d_bytes"], S.nbytes + E.nbytes + st["d2h_bytes"], float(E.mean())

    e2e_step(0)
    rt.barrier()
    e2e_t, n_e2e = 0.0, steps
    for k in range(n_e2e):
        dt, h2d, d2h, Emean = e2e_step(warmup + k)
        e2e_t += dt
    rt.barrier()
    t_e2e = rt.max_over_ranks(e2e_t)
    upd_step = N_SITES * REPLICAS * sweeps
    if rt.rank != 0:
        return None
    pk = peaks()
    kern_s = float(np.mean([s["kernel_ms"] for s in stats])) / 1e3
    flips = float(np.mean([s["flips"] for s in stats]))
    alg_bytes = flips * N_SITES * bJ
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    smem_peak = 128.0 * rt.sms * sm_mhz * 1e6 / 1e9      # GB/s: 128 B/clk/SM at the clock seen in the timed region
    achieved = alg_bytes / kern_s / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("ssf_kernel_dram_bytes_per_launch")
    line = base_line(upd_step * steps * rt.world / t_dev, rt.world, steps, warmup, 1e3 * t_dev / steps, prec_name, c2_config(args))
    line["roofline"] = {
        "bound": "smem", "achieved": achieved, "peak": smem_peak, "unit": "GB/s", "frac": achieved / smem_peak,
        "traffic": traffic, "kernel": "isb::ssf_kernel (streaming and plain instantiations) + isb::ssf_cold_kernel, one per segment of the anneal",
        "kernel_ms": 1e3 * kern_s,
        "peak_source": f"shared-memory / L1 data path, 128 B/clk/SM x {rt.sms} SMs x {sm_mhz:.0f} MHz (clock sampled in the timed region)",
        "accounting": f"row bytes the chains read through the SM's shared-memory / L1 data path: accepted flips ({flips:.4g} per "
                      f"anneal) x N x {bJ} B (one J row per accepted flip per chain: 128-bit LDS from the ring while the streaming "
                      "kernel runs, 128-bit loads that hit L1 / L2 once the plain kernel has taken over); ring writes of the "
                      "streamed epochs not counted",
        "accept_rate": flips / upd_step,
        "launches_per_anneal": float(np.mean([s["launches"] for s in stats])),
        "traffic_note": "DRAM bytes of ONE launch of the sweep kernel (ncu); an anneal is run as several launches (streaming kernel "
                        "while hot, plain kernel once cold), each of which reads the cached fields and spins once",
        "hbm_accounting": {"note": "SURVEY §8d per-chain figure (flips x N x b_J) against the measured HBM copy rate: > 1 because "
                                   "one smem copy of a row serves all chains of a CTA; DRAM traffic is ~46 MB per launch, so "
                                   "the HBM roof (and the >= 60 % HBM target) is moot for this design",
                           "GBps": achieved, "hbm_peak_GBps": pk["hbm"], "ratio": achieved / pk["hbm"],
                           "attempts_accounting_GBps": upd_step * N_SITES * bJ / kern_s / 1e9}}
    line["e2e"] = {"value": upd_step * n_e2e * rt.world / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                   "d2h_bytes_per_step": int(d2h), "mean_final_energy": Emean}
    line["gpu_launches"] = int(sum(s["launches"] for s in stats))
    line["clocks"] = clocks
    if cpu and rt.world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baselines(lambda s, t=None: c2_cpu_rate(sweeps, s, t), args.cpu_seconds)
    return line


# ---------------------------------------------------------------------------------------------- C1: 32x32 lattice
def c1_config(args):
    sweeps = args.c1_sweeps
    return {"workload": f"C1: 32x32 periodic ferromagnet (sparse J, 4 neighbours), Metropolis at T=2.269, {sweeps} sequential "
                        f"sweeps, 4096 replicas/GPU", "n_sites": 1024, "replicas_per_gpu": 4096, "sweeps_per_step": sweeps,
            "updates_per_step_per_gpu": 1024 * 4096 * sweeps, "sharding": "replicas (no collective)", "l2": "flushed between timed steps"}


def run_c1(rt, args, steps, warmup, cpu=True, dump=None):
    """BASELINE config 1: built from a sparse J exactly as the reference's tests / demo build theirs."""
    import scipy.sparse as sp
    from isingmodel_jl_b200 import synth, SpinSystems, SingleSpinFlip, SamplingHelper
    L = rt.L
    N, R, T1 = 1024, 4096, 2.269
    sweeps = args.c1_sweeps
    J = sp.csc_matrix(synth.lattice_J(32))
    nsteps = sweeps * N
    upd_step = N * R * sweeps
    pin = rt.pinned((R, N))
    pin[:] = synth.spins(SEED_S + 1000 * rt.rank, R, N)
    ss = SpinSystems.SpinSystem(pin, J, np.zeros(N), device=rt.local)
    ua = SingleSpinFlip.MetropolisMethod(ss, T1)
    ens = ss._ensemble()
    rt.last_stats = ens.last_stats
    Tarr = np.array([T1])
    last = {}

    def step(k):
        last["out"] = ens.ssf_run(L.RULE_METROPOLIS, nsteps, seed=99 + rt.rank, step_offset=k * nsteps, T=Tarr,
                                  steps_per_T=nsteps)

    steps, t_dev, stats, clocks = rt.run_steps(lambda: ens.set_spins(pin), step, warmup, steps)
    if dump and rt.rank == 0:
        dump_outputs(dump, {"spins": ens.get_spins(), "flips": last["out"]["flips"]})
    rt.barrier()
    n_e2e = min(steps, 5)
    t0 = time.perf_counter()
    for k in range(n_e2e):
        ss.spinConfiguration = pin
        SamplingHelper.run_(ua, nsteps, order="sequential", seed=99 + rt.rank, step_offset=(warmup + k) * nsteps,
                            temperatures=Tarr, steps_per_T=nsteps)
        S = ss.spinConfiguration
        E = SpinSystems.calcEnergy(ua)
    rt.torch.cuda.synchronize()
    t_e2e = rt.max_over_ranks(time.perf_counter() - t0)
    # R = 1 latency: config 1 is "the reference CPU path" — ONE chain; the time per sweep of a single chain is what a
    # user of the reference's one SpinSystem sees
    ss1 = SpinSystems.SpinSystem(pin[:1].copy(), J, np.zeros(N), device=rt.local)
    e1 = ss1._ensemble()
    lat_sweeps = min(sweeps, 2000)
    for _ in range(2):
        e1.set_spins(pin[:1])
        e1.ssf_run(L.RULE_METROPOLIS, lat_sweeps * N, seed=7, T=Tarr, steps_per_T=lat_sweeps * N)
    lat_ms = e1.last_stats()["kernel_ms"]
    # beside the reference's sequential sweep: the two-colour sweep order (ISB_ORDER_CHECKERBOARD, SURVEY §8f rank 1 — one
    # particular site list of the 3-argument update!, executed 32 sites at a time), same model, same rule, same noise words
    cb = {}
    for name, eX, reps in (("all_replicas", ens, 1), ("single_chain", e1, 2)):
        sw = sweeps if name == "all_replicas" else lat_sweeps
        for _ in range(1 + reps):
            eX.set_spins(pin if name == "all_replicas" else pin[:1])
            eX.ssf_run(L.RULE_METROPOLIS, sw * N, order=L.ORDER_CHECKERBOARD, seed=7, T=Tarr, steps_per_T=sw * N)
        cb[name] = (sw, eX.last_stats()["kernel_ms"])
    cb_Emean = float(ens.energy().mean())
    if rt.rank != 0:
        return None
    kern_s = float(np.mean([s["kernel_ms"] for s in stats])) / 1e3
    flips = float(np.mean([s["flips"] for s in stats]))
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    line = base_line(upd_step * steps * rt.world / t_dev, rt.world, steps, warmup, 1e3 * t_dev / steps, "f64", c1_config(args))
    # issue-slot roofline: no J streaming at all (4 neighbours per site, spins as bits in shared memory), the kernel is bound
    # by the instructions it issues; the count per 32-site window comes from ncu (profiles/) and the peak is
    # 4 warp-instructions / clk / SM
    ipu = C1_INSTR_PER_UPDATE
    issue_peak = 4.0 * 32.0 * rt.sms * sm_mhz * 1e6 / ipu          # updates/s at 100 % issue utilisation
    line["roofline"] = {"bound": "issue", "achieved": upd_step / kern_s, "peak": issue_peak, "unit": "updates/s",
                        "frac": upd_step / kern_s / issue_peak, "traffic": None, "kernel": C1_KERNEL, "kernel_ms": 1e3 * kern_s,
                        "accept_rate": flips / upd_step,
                        "accounting": f"issue slots: {ipu} warp instructions per 32-site window of a chain (ncu count of the committed "
                                      f"kernel, profiles/r2o_c1_lattice_ncu_summary.txt) at 4 warp-instructions/clk/SM x {rt.sms} SMs x "
                                      f"{sm_mhz:.0f} MHz; the working set of a chain is on chip: no HBM traffic in steady state",
                        "hbm_accounting_GBps": flips * 4 * 12.0 / kern_s / 1e9}
    tb, tsrc = captured_traffic("ssf_lattice_kernel_c1_per_300_sweep_launch")
    if tb:
        line["roofline"].update({"traffic": tb, "traffic_source": tsrc + "; independent of the sweep count (spins in, bits on chip)"})
    line["e2e"] = {"value": upd_step * n_e2e * rt.world / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(pin.nbytes),
                   "d2h_bytes_per_step": int(S.nbytes + E.nbytes), "mean_final_energy": float(E.mean()),
                   "exact_mean_energy_kaufman": -1468.4}
    line["single_chain_latency"] = {"replicas": 1, "sweeps": lat_sweeps, "kernel_ms": lat_ms,
                                    "us_per_sweep": 1e3 * lat_ms / lat_sweeps, "updates_per_s": lat_sweeps * N / (lat_ms / 1e3)}
    line["checkerboard_order"] = {
        "note": "NOT the headline: the same model and rule swept in two-colour order (all sites with x + y even, then the others) "
                "instead of the reference's sequential site order; bit-exact with the oracle walking that site list "
                "(tests/test_gpu_lattice.py), kernel isb::ssf_lattice_cb_kernel",
        "value": N * R * cb["all_replicas"][0] / (cb["all_replicas"][1] / 1e3), "unit": UNIT, "kernel_ms": cb["all_replicas"][1],
        "mean_final_energy": cb_Emean,
        "single_chain_us_per_sweep": 1e3 * cb["single_chain"][1] / cb["single_chain"][0]}
    line["gpu_launches"] = int(sum(s["launches"] for s in stats))
    line["clocks"] = clocks
    if cpu and rt.world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baselines(lambda s, t=None: c1_cpu_rate(s, t), args.cpu_seconds)
    return line


# C1's dominant kernel and the warp instructions it executes per 32-site window (= thread-instructions per update with all
# 32 lanes counted): ncu of the committed kernel, 14 617 209 657 warp instructions / 39 321 600 windows
# (profiles/r2o_c1_lattice_ncu_summary.txt)
C1_KERNEL = "isb::ssf_lattice_kernel"
C1_INSTR_PER_UPDATE = 371.7


# ---------------------------------------------------------------------------------------------- C3 / C4: contractions
SCA_STEPS = {"c3": 200, "c4": 1000}


def sca_workload(which):
    """(W, h_visible, b_hidden, R, T schedule factory, description) of BASELINE.json configs[2] / configs[3]."""
    from isingmodel_jl_b200 import synth
    if which == "c4":
        W, h, b = synth.bipartite_W(784, 512, 4, 0.1)
        return W, h, b, 16384, (lambda n: np.ones(n)), "C4: bipartite 784x512 block Gibbs (SCA), 16384 chains/GPU, T=1"
    N = 4096
    J = synth.sk_J(N, 3)
    # pinning parameter q = eigmax(J)/2 (demo.jl:82); W = (J + qI)/2, biases h/2 (h = 0 here)
    q = 0.5 * float(np.linalg.eigvalsh(J)[-1])
    W = 0.5 * (J + q * np.eye(N))
    z = np.zeros(N)
    return W, z, z, 8192, (lambda n: np.linspace(1.0, 0.05, n)), \
        f"C3: dense Gaussian J N=4096 MultiSpinFlip SCA (bipartite embedding W=(J+qI)/2, q={q:.4f}), 8192 replicas/GPU, linear annealing T 1->0.05"


def sca_config(which, desc, W, R, nst, prec_name=None):
    nv, nh = W.shape
    c = {"workload": desc + f", {nst} SCA steps per bench step", "nv": nv, "nh": nh, "chains_per_gpu": R,
         "sca_steps_per_step": nst, "updates_per_step_per_gpu": (nv + nh) * R * nst,
         "sharding": "replicas (no collective)",
         "l2": "flushed between timed steps (256 MiB write); the spin matrices are re-read every half-step, W is L2-resident"}
    if prec_name:
        c["coupling_storage"] = prec_name
    return c


def run_sca(rt, args, which, precs, steps, warmup, cpu=True, dump=None):
    """precs[0] is the primary precision (top level of the result, with e2e); the others are timed the same way and
    reported under `precisions`."""
    from isingmodel_jl_b200 import synth, SpinSystems, OnBipartiteGraph, SamplingHelper
    L = rt.L
    nst = args.sca_steps or SCA_STEPS[which]
    W, h, b, R, sched, desc = sca_workload(which)
    nv, nh = W.shape
    T = sched(nst)
    upd_step = (nv + nh) * R * nst
    pv, ph = rt.pinned((R, nv)), rt.pinned((R, nh))
    pv[:] = synth.spins(11 + 1000 * rt.rank, R, nv)
    ph[:] = synth.spins(12 + 1000 * rt.rank, R, nh)
    pk = peaks()
    out = None
    for i, prec_name in enumerate(precs):
        prec = {"bf16x3": L.PREC_BF16X3, "bf16x2": L.PREC_BF16X2, "bf16x1": L.PREC_BF16X1, "f64": L.PREC_F64,
                "fp16x2": L.PREC_FP16X2, "fp16x1": L.PREC_FP16X1, "i8x3": L.PREC_I8X3, "i8x2": L.PREC_I8X2,
                "i8x4": L.PREC_I8X4}[prec_name]
        P = PREC_PASSES[prec_name]
        ss = SpinSystems.SpinSystemOnBipartiteGraph(pv, ph, W, h, b, device=rt.local, prec=prec)
        ua = OnBipartiteGraph.StochasticCellularAutomata(ss, float(T[0]))
        ens = ss._ensemble()
        rt.last_stats = ens.last_stats

        def reset():
            ens.set_spins(pv)
            ens.set_hidden(ph)

        def step(k):
            ens.bip_run(L.BIP_SCA, nst, seed=777 + rt.rank, step_offset=k * nst, T=T)

        nsteps_i, t_dev, stats, clocks = rt.run_steps(reset, step, warmup, steps if i == 0 else None)
        e2e = None
        if i == 0:
            if dump and rt.rank == 0:
                dump_outputs(dump, {"spins": ens.get_spins(), "hidden": ens.get_hidden()})
            def e2e_step(k):
                rt.flush.zero_()
                rt.torch.cuda.synchronize()
                t0 = time.perf_counter()
                ss.spinConfiguration = pv
                ss.hiddenLayer = ph
                SamplingHelper.run_(ua, nst, seed=777 + rt.rank, step_offset=k * nst, temperatures=T)
                st = ens.last_stats()
                S, Tm = ss.spinConfiguration, ss.hiddenLayer
                E = SpinSystems.calcEnergy(ua)
                rt.torch.cuda.synchronize()
                return (time.perf_counter() - t0, pv.nbytes + ph.nbytes + st["h2d_bytes"],
                        S.nbytes + Tm.nbytes + E.nbytes + st["d2h_bytes"], float(E.mean()))
            e2e_step(0)
            rt.barrier()
            n_e2e, e2e_t = min(nsteps_i, 5), 0.0
            for k in range(n_e2e):
                dt, h2d, d2h, Emean = e2e_step(warmup + k)
                e2e_t += dt
            rt.barrier()
            t_e2e = rt.max_over_ranks(e2e_t)
            v_e2e, v_dev = upd_step * n_e2e * rt.world / t_e2e, upd_step * nsteps_i * rt.world / t_dev
            e2e = {"value": v_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                   "mean_final_energy": Emean, "steps": n_e2e, "frac_of_device_value": v_e2e / v_dev}
        del ua, ss, ens
        if rt.rank != 0:
            continue
        kern_s = float(np.mean([s["kernel_ms"] for s in stats])) / 1e3 / (2 * nst)   # average half-step
        alg = 2.0 * nv * nh * R                                                        # algorithmic flops per half-step
        ach = alg / kern_s / 1e12
        res = base_line(upd_step * nsteps_i * rt.world / t_dev, rt.world, nsteps_i, warmup, 1e3 * t_dev / nsteps_i,
                        "f64" if prec_name == "f64" else ("i8" if prec_name.startswith("i8") else prec_name[:4]),
                        sca_config(which, desc, W, R, nst, prec_name))
        peak, peak_src = tensor_peak(pk, t_dev)
        res["roofline"] = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                           "traffic": None, "peak_source": peak_src,
                           "kernel": "isb::bip_tc_kernel", "kernel_ms_per_half_step": 1e3 * kern_s,
                           "passes_bf16_equivalent": P, "executed_TFLOPs_bf16_equivalent": ach * P,
                           "executed_frac": ach * P / peak,
                           "peak_burst": pk["tc_burst"], "frac_of_burst": ach / pk["tc_burst"],
                           "peak_sustained": pk["tc_sustained"], "frac_of_sustained": ach / pk["tc_sustained"],
                           "timed_region_s": t_dev,
                           "accounting": "algorithmic = 2 x N_out x N_in x R flop per half-step (the contraction of the reference's "
                                         "W'sigma / W tau, once); executed = passes x algorithmic in bf16-pass equivalents "
                                         "(an int8 pass runs at twice the bf16 tensor rate and moves half the bytes)",
                           "storage": PREC_NOTE[prec_name]}
        if prec_name == "i8x3":
            launches_per_step = float(np.mean([s["launches"] for s in stats]))
            if which == "c3" and launches_per_step == 2 * nst:          # one launch per half-step, as captured
                tb, tsrc = captured_traffic("bip_tc_kernel_c3_i8x3_per_half_step_launch")
                if tb:
                    res["roofline"].update({"traffic": tb, "traffic_source": tsrc})
            elif which == "c4" and launches_per_step == 1:              # chain-resident: one launch per bench step
                tb, tsrc = captured_traffic("bip_tc_kernel_c4_i8x3_per_100_step_launch")
                if tb:
                    res["roofline"].update({"traffic": tb * nst / 100.0, "traffic_source": tsrc + f"; scaled from 100 to {nst} SCA steps per launch"})
        res["gpu_launches"] = int(sum(s["launches"] for s in stats))
        res["clocks"] = clocks
        if e2e:
            res["e2e"] = e2e
        if out is None:
            out = res
            out["precisions"] = {}
        else:
            out["precisions"][prec_name] = {k: res[k] for k in ("value", "steps", "ms_per_step", "dtype", "roofline", "clocks", "gpu_launches")}
    if rt.rank != 0:
        return None
    if cpu and rt.world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baselines(lambda s, t=None: sca_cpu_rate(W, h, b, T, s, t), args.cpu_seconds)
    return out


# ---------------------------------------------------------------------------------------------- C5: row-sharded SCA
def run_c5(rt, args, prec_name, steps, warmup, dump=None):
    """BASELINE config 5: dense J with N = 8192 x GPUs (65536 on 8), rows of W = (J + qI)/2 sharded across the GPUs,
    R replicas, SCA annealing, the freshly sampled spin blocks exchanged after every half-step (NVLink)."""
    from isingmodel_jl_b200 import synth, rowshard
    L = rt.L
    prec = {"bf16x3": L.PREC_BF16X3, "bf16x2": L.PREC_BF16X2, "bf16x1": L.PREC_BF16X1, "i8x3": L.PREC_I8X3,
            "i8x2": L.PREC_I8X2, "i8x4": L.PREC_I8X4}[prec_name]
    P = PREC_PASSES[prec_name]
    esz = 1 if prec_name.startswith("i8") else 2
    nb, R = args.c5_n_per_gpu, args.c5_replicas
    n = nb * rt.world
    nst = args.sca_steps or 10
    # default: the step loop inside the library (isb_shard_run_*, the C-ABI entry of this path) with the copy-engine
    # exchange; ISB_C5_EXCHANGE = abi-nccl | copy | nccl | pipelined | fused selects the alternatives (the last four
    # drive the half-steps from Python over torch: the round-1 host loop)
    ex = os.environ.get("ISB_C5_EXCHANGE") or "abi-copy"
    if ex.startswith("abi-") or rt.world == 1:
        sca = rowshard.ShardRunSCA(n, R, seed=5, q=1.0, prec=prec, device=rt.local, exchange=ex[4:] if ex.startswith("abi-") else "copy")
    else:
        sca = rowshard.RowShardedSCA(n, R, seed=5, q=1.0, prec=prec, device=rt.local, exchange=ex)
    S0 = synth.spins(21, R, n)   # the same initial configuration on every rank
    T = np.linspace(1.0, 0.05, nst)
    rt.last_stats = lambda: {}
    l0 = sca.launches

    def step(k):
        sca.run(nst, T, seed=31, step_offset=k * nst)

    steps, t_dev, _, clocks = rt.run_steps(lambda: sca.set_spins(S0), step, warmup, steps)
    if dump and rt.rank == 0:
        dump_outputs(dump, {"spins": sca.get_spins()})
    launches = (sca.launches - l0) * steps // (steps + warmup)
    pin = rt.pinned((R, n))
    pin[:] = S0
    rt.barrier()
    n_e2e = min(steps, 3)
    t0 = time.perf_counter()
    for k in range(n_e2e):
        sca.set_spins(pin)
        sca.run(nst, T, seed=31, step_offset=(warmup + k) * nst)
        out = sca.get_spins()
    rt.torch.cuda.synchronize()
    t_e2e = rt.max_over_ranks(time.perf_counter() - t0)
    upd_step = 2 * n * R * nst
    exchange = sca.exchange
    del sca
    if rt.rank != 0:
        return None
    pk = peaks()
    half_s = t_dev / steps / (2 * nst)
    flops = 2.0 * nb * n * R            # per GPU per half-step (algorithmic)
    gather = (rt.world - 1) * R * nb * esz   # bytes received per GPU per half-step
    peak, peak_src = tensor_peak(pk, t_dev)
    t_mma, t_link = flops * P / (peak * 1e12), gather / 770e9
    ach = flops / half_s / 1e12
    nccl_lines = []
    if rt.nccl_log:
        import glob
        for path in sorted(glob.glob(rt.nccl_log + "*")):
            for ln in open(path, errors="replace"):
                if any(key in ln for key in ("nranks", "NVLS", "Connected all", "Init COMPLETE", "NCCL version", "via P2P", "via NVL")):
                    nccl_lines.append(ln.strip()[-220:])
        if len(nccl_lines) > 8:
            nccl_lines = nccl_lines[:6] + nccl_lines[-2:]
    cfg = {"workload": f"C5: dense SK J N={n} row-sharded over {rt.world} GPU(s) ({nb} rows each), {R} replicas, "
                       f"SCA annealing T 1->0.05, {nst} steps per bench step, spin blocks exchanged after every half-step",
           "n": n, "rows_per_gpu": nb, "replicas": R, "coupling_storage": prec_name,
           "collective": {"abi-copy": "inside the library (isb_shard_run_steps): copy-engine pushes into the peers' gathered matrices over "
                                      "CUDA IPC + stream memory operations, hidden under the other replica group's GEMM",
                          "abi-nccl": "inside the library (isb_shard_run_steps): ncclAllGather per half-step on a side stream, hidden "
                                      "under the other replica group's GEMM",
                          "pipelined": "ncclAllGather per half-step, hidden under the other replica group's GEMM",
                          "nccl": "ncclAllGather per half-step (torch.distributed)",
                          "copy": "copy-engine pushes into symmetric memory + barrier, hidden under the other replica group's GEMM",
                          "fused": "peer stores fused into the sampling epilogue (symmetric memory) + barrier",
                          "local": "none (1 GPU)"}[exchange],
           "exchange": exchange, "l2": "flushed between timed steps; W block (>= 1 GiB) exceeds L2"}
    res = base_line(upd_step * steps / t_dev, rt.world, steps, warmup, 1e3 * t_dev / steps, "i8" if esz == 1 else "bf16", cfg)
    res["scaling"] = "weak (N grows with the GPU count: 8192 rows of J per GPU)"
    res["roofline"] = {"bound": "tensor" if t_mma >= t_link else "nvlink", "achieved": ach, "peak": peak,
                       "unit": "TFLOP/s", "frac": ach / peak, "traffic": None, "peak_source": peak_src, "kernel": "isb::bip_tc_kernel",
                       "kernel_ms_per_half_step": 1e3 * half_s, "passes_bf16_equivalent": P, "executed_frac": ach * P / peak,
                       "peak_burst": pk["tc_burst"], "frac_of_burst": ach / pk["tc_burst"],
                       "peak_sustained": pk["tc_sustained"], "frac_of_sustained": ach / pk["tc_sustained"], "timed_region_s": t_dev,
                       "fused_target_ms": 1e3 * max(t_mma, t_link),
                       "fused_target": "max(passes x flops / the cuBLAS bf16 rate named in peak_source, exchanged bytes / 770 GB/s)",
                       "frac_of_fused_target": max(t_mma, t_link) / half_s, "mma_only_ms": 1e3 * t_mma, "link_only_ms": 1e3 * t_link,
                       "exchanged_bytes_per_gpu_per_half_step": gather, "storage": PREC_NOTE[prec_name]}
    res["e2e"] = {"value": upd_step * n_e2e / t_e2e, "unit": UNIT, "h2d_bytes_per_step": int(pin.nbytes),
                  "d2h_bytes_per_step": int(out.nbytes), "steps": n_e2e}
    res["gpu_launches"] = int(launches)
    res["clocks"] = clocks
    res["nccl"] = nccl_lines
    return res


# ---------------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (default 10: a C2 step is 195 ms, so the timed region is 2 s)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--sweeps", type=int, default=1000, help="c2: annealing sweeps per step (SURVEY §8d C2: 1000)")
    ap.add_argument("--c1-sweeps", type=int, default=10000, help="c1: sweeps per step (BASELINE configs[0]: 10^4)")
    ap.add_argument("--ref-seconds", type=float, default=4.0, help="CPU seconds per reference-arm step")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="CPU seconds of each cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--prec", default=None,
                    help="c2: f64 | f32; c3/c4/c5: i8x3 (default) | i8x2 | i8x4 | fp16x2 | bf16x3 | bf16x2 | bf16x1 | f64; "
                         "a comma list times several (the first is the primary)")
    ap.add_argument("--c5-n-per-gpu", type=int, default=8192, help="c5: rows of J per GPU (N = this x GPUs; 8 GPUs -> 65536)")
    ap.add_argument("--c5-replicas", type=int, default=1024)
    ap.add_argument("--workload", default="all", choices=["all", "c1", "c2", "c3", "c4", "c5"],
                    help="all (default): the C2 headline + every other BASELINE config as `workloads` sub-results")
    ap.add_argument("--sca-steps", type=int, default=None, help="SCA steps per bench step (c3: 200, c4: 1000, c5: 10)")
    ap.add_argument("--sub-warmup", type=int, default=3, help="warm-up steps of the sub-workloads")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the printed workload computed as DIR/<name>.npy (rank 0's replicas)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times bounded samples and has no outputs to compare")
    # ONE JSON line on stdout: whatever a library prints there (NCCL's version banner under NCCL_DEBUG, compiler chatter)
    # is sent to stderr at the file-descriptor level; the line itself goes to the saved descriptor at the end
    out = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    if args.impl == "reference":
        return reference_arm(args, out)

    rt = Runtime(args)
    tensor_precs = args.prec.split(",") if args.prec and args.workload != "c2" else ["i8x3", "fp16x2", "bf16x3", "bf16x1"]
    c5_prec = tensor_precs[0] if tensor_precs[0] in ("bf16x3", "bf16x2", "bf16x1", "i8x3", "i8x2", "i8x4") else "i8x3"
    dump = args.dump_outputs
    if args.workload == "c2":
        line = run_c2(rt, args, args.steps, args.warmup, dump=dump)
    elif args.workload == "c1":
        line = run_c1(rt, args, args.steps, args.warmup, dump=dump)
    elif args.workload in ("c3", "c4"):
        line = run_sca(rt, args, args.workload, tensor_precs, args.steps, args.warmup, dump=dump)
    elif args.workload == "c5":
        line = run_c5(rt, args, c5_prec, args.steps, args.warmup, dump=dump)
    else:
        line = run_c2(rt, args, args.steps, args.warmup, dump=dump)
        subs = {}
        if rt.world == 1:
            subs["c1"] = run_c1(rt, args, None, args.sub_warmup)
            subs["c3"] = run_sca(rt, args, "c3", tensor_precs, None, args.sub_warmup)
            subs["c4"] = run_sca(rt, args, "c4", tensor_precs, None, args.sub_warmup)
        else:
            # the one path with a real exchange step; the replica-sharded configs (c1, c3, c4) scale like the headline
            # (no collective) and are measured at N = 1
            subs["c5"] = run_c5(rt, args, c5_prec, None, args.sub_warmup)
            alt = run_c5(rt, args, "bf16x3", None, args.sub_warmup) if c5_prec != "bf16x3" else None
            if rt.rank == 0 and alt:
                subs["c5"]["precisions"] = {"bf16x3": {k: alt[k] for k in ("value", "steps", "ms_per_step", "roofline", "clocks", "e2e")}}
        if rt.rank == 0:
            line["workloads"] = subs
    if rt.rank == 0:
        out.write(json.dumps(line) + "\n")
        out.flush()
    rt.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
