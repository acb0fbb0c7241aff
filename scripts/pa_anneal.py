"""Population annealing on C2's workload (SK N = 1024, Glauber, geometric 2.0 -> 0.05) and on C1's lattice (32 x 32 torus,
Metropolis, geometric 5.0 -> 2.269), 4096 replicas in one population, --steps temperature steps x --sweeps sweeps each
(default 200 x 5 = C2's 1000 sweeps).  Prints one JSON document (and writes it to --out).

Per model:
  (a) device time of one isb_ssf_run_pa call against the same per-step traced isb_ssf_run calls without resampling
      (isb_ens_last_stats of each call), which isolates the cost of the resampling;
  (b) the resampling and gather kernels' time per temperature step, from torch.profiler in a separate run;
  (c) a host-driven population annealing (traced isb_ssf_run per step, numpy systematic resampling, get_spins /
      set_spins) against tempering.PopulationAnnealing, wall clock per anneal (both end in a device synchronisation);
  (d) surviving families and the final <E>/N of the device anneal.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
    import torch
    info = {"torch_device": torch.cuda.get_device_name(0)}
    try:   # read-only query
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except (OSError, subprocess.TimeoutExpired) as exc:
        info["nvidia_smi"] = f"unavailable: {exc}"
    return info


def system(kind, R, steps):
    import scipy.sparse as sp
    from isingmodel_jl_b200 import SingleSpinFlip, SpinSystems, synth
    N = 1024
    if kind == "c2":
        ss = SpinSystems.SpinSystem(synth.spins(3, R, N), synth.sk_J(N, 2), np.zeros(N))
        return ss, SingleSpinFlip.GlauberDynamics(ss, 1.0), np.geomspace(2.0, 0.05, steps)
    ss = SpinSystems.SpinSystem(synth.spins(3, R, N), sp.csc_matrix(synth.lattice_J(32)), np.zeros(N))
    return ss, SingleSpinFlip.MetropolisMethod(ss, 1.0), np.geomspace(5.0, 2.269, steps)


def host_pa(ens, rule, T, spt, seed):
    """Population annealing driven from the host: one traced isb_ssf_run per temperature, systematic resampling in numpy
    (one population), the selected spins uploaded with set_spins (which rebuilds the cached fields)."""
    R, n = ens.R, ens.nv
    rng = np.random.default_rng(seed)
    fam = np.arange(R)
    for k in range(len(T)):
        out = ens.ssf_run(rule, spt, start=(k * spt) % n, seed=seed, step_offset=k * spt, T=np.array([T[k]]),
                          steps_per_T=spt, trace_every=spt, want_M=False)
        if k + 1 < len(T):
            a = -(1.0 / T[k + 1] - 1.0 / T[k]) * out["E"][0]
            w = np.exp(a - a.max())
            C = np.cumsum(w)
            parent = np.minimum(np.searchsorted(C, (np.arange(R) + rng.random()) * C[-1] / R, side="right"), R - 1)
            ens.set_spins(ens.get_spins()[parent])
            fam = fam[parent]
    return out["E"][0], fam


def measure(kind, args):
    import torch
    from isingmodel_jl_b200 import _lib as L, tempering
    R, N = 4096, 1024
    spt = args.sweeps * N
    res = {"model": {"c2": "SK N=1024 dense Gaussian J, Glauber, T 2.0 -> 0.05",
                     "c1": "32x32 periodic ferromagnet (sparse J), Metropolis, T 5.0 -> 2.269"}[kind],
           "replicas": R, "populations": 1, "temperature_steps": args.steps, "sweeps_per_step": args.sweeps}

    # (c) and (d): the device class against the host-driven loop, wall clock per whole anneal
    dev_s, host_s = [], []
    for rep in range(args.reps + 1):            # the first anneal of each is a warm-up
        ss, ua, T = system(kind, R, args.steps)
        pa = tempering.PopulationAnnealing(ua, seed=1)
        ens = ss._ensemble()
        torch.cuda.synchronize()
        t = time.perf_counter()
        E = pa.run(T, sweeps=args.sweeps)
        dt = time.perf_counter() - t
        if rep:
            dev_s.append(dt)
        st = ens.last_stats()
        fs = pa.family_statistics()
        res["device_anneal"] = {"pa_call_device_ms": st["kernel_ms"], "launches": st["launches"],
                                "families": int(fs["families"][0]), "rho_t": float(fs["rho_t"][0]),
                                "family_entropy": float(fs["entropy"][0]), "final_mean_E_per_site": float(E[-1].mean() / N),
                                "lnZ_final_over_first": float(pa.lnZ[0])}
        ss2, ua2, _ = system(kind, R, args.steps)
        ens2 = ss2._ensemble()
        torch.cuda.synchronize()
        t = time.perf_counter()
        Eh, famh = host_pa(ens2, ua2._rule, T, spt, 1)
        dt = time.perf_counter() - t
        if rep:
            host_s.append(dt)
        res["host_anneal"] = {"families": int(len(np.unique(famh))), "final_mean_E_per_site": float(Eh.mean() / N)}
    res["device_anneal"]["wall_s"] = dev_s
    res["host_anneal"]["wall_s"] = host_s
    res["speedup_wall_median"] = float(np.median(host_s) / np.median(dev_s))

    # (a) the same per-step traced sweeps without resampling, on a fresh ensemble from the same start
    ss, ua, T = system(kind, R, args.steps)
    ens = ss._ensemble()
    ms = 0.0
    for k in range(args.steps):
        ens.ssf_run(ua._rule, spt, start=(k * spt) % N, seed=1, step_offset=k * spt, T=np.array([T[k]]), steps_per_T=spt,
                    trace_every=spt, want_M=False)
        ms += ens.last_stats()["kernel_ms"]
    pa_ms = res["device_anneal"]["pa_call_device_ms"]
    res["sweeps_alone_device_ms"] = ms
    res["pa_device_ms_over_sweeps_alone"] = pa_ms / ms
    res["resampling_device_us_per_step"] = 1e3 * (pa_ms - ms) / max(args.steps - 1, 1)

    # (b) kernel totals of a separate, profiled anneal
    from torch.profiler import ProfilerActivity, profile
    ss, ua, T = system(kind, R, args.steps)
    pa = tempering.PopulationAnnealing(ua, seed=1)
    ss._ensemble()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        pa.run(T, sweeps=args.sweeps)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        if us > 0:
            kern[ev.key[:90]] = {"calls": ev.count, "total_us": us}
    resample_us = sum(v["total_us"] for k, v in kern.items() if "pa_" in k or "gather_rows" in k)
    gather_us = sum(v["total_us"] for k, v in kern.items() if "gather_rows" in k)
    res["profiled"] = {"kernels": kern, "resample_and_gather_us_per_step": resample_us / max(args.steps - 1, 1),
                       "gather_us_per_step": gather_us / max(args.steps - 1, 1)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--sweeps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--models", default="c2,c1")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("pa_anneal.py measures on a CUDA device; none is visible")
    doc = {"card": card(), "args": {k: v for k, v in vars(args).items() if k != "out"}, "results": {}}
    for kind in args.models.split(","):
        doc["results"][kind] = measure(kind, args)
        print(kind, json.dumps(doc["results"][kind]), flush=True)
    doc["card_after"] = card()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
