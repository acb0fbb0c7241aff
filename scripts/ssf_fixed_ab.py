"""The fixed-point dense sweep kernels against the Float64 ones on the C2 anneal (SK N = 1024, 4096 replicas, Glauber,
1000 sweeps of bench.py's geometric schedule, Philox noise).  Prints one JSON document (and writes it to --out).

- anneal: device time (isb_ens_last_stats) of whole anneals on each path (ISB_SSF_FIXED = 1 / 0), each starting from
  set_spins (so each includes one field initialisation), flips and exact fallbacks per anneal;
- field_init_ms: one field initialisation of each path (a 1-step run after set_spins minus a 1-step run without);
- profile: the anneal cut into 50-sweep chunks; every chunk is run from the same state with each kernel forced
  (ISB_SSF_MODE = 2 streaming, Float64 only since the fixed-point path has no streaming kernel; 1 plain; 0 cold), timed
  without the field initialisation, with its acceptance.  The chunk's fastest kernel against its acceptance is what the segment thresholds of ssf_run_device are read from;
- thresholds: whole fixed-point anneals under a grid of ISB_SSF_COLD_THR."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

N, R, SWEEPS, CHUNK = 1024, 4096, 1000, 50


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--thr", default="0.02,0.025,0.03,0.035,0.045,0.06", help="ISB_SSF_COLD_THR values of the grid")
    args = ap.parse_args()
    import bench
    from isingmodel_jl_b200 import _lib as L, synth
    J, h, T = bench.workload(SWEEPS)
    S0 = synth.spins(bench.SEED_S, R, N)
    ctx = L.context(0)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    res = {"card": card(), "model": f"SK N = {N}, {R} replicas, Glauber, {SWEEPS} sweeps"}

    def run(nsteps, t0=0, fixed=True):
        os.environ["ISB_SSF_FIXED"] = "1" if fixed else "0"
        e.ssf_run(L.RULE_GLAUBER, nsteps, start=t0 % N, seed=12345, step_offset=t0, T=T[t0 // N:], steps_per_T=N)
        return e.last_stats()

    anneal = {"fixed": [], "float64": []}
    for rep in range(args.reps + 1):
        for path in ("fixed", "float64"):
            e.set_spins(S0)
            st = run(SWEEPS * N, fixed=path == "fixed")
            if rep > 0:
                anneal[path].append({k: st[k] for k in ("kernel_ms", "launches", "flips", "exact_fallbacks")})
    res["anneal"] = anneal
    res["anneal_ms_median"] = {p: float(np.median([a["kernel_ms"] for a in v])) for p, v in anneal.items()}

    init = {}
    for path in ("fixed", "float64"):
        with_init, without = [], []
        for _ in range(5):
            e.set_spins(S0)
            with_init.append(run(1, fixed=path == "fixed")["kernel_ms"])
            without.append(run(1, t0=1, fixed=path == "fixed")["kernel_ms"])
        init[path] = float(np.median(with_init) - np.median(without))
    res["field_init_ms"] = init

    prof = {"fixed": [], "float64": []}
    for path in ("fixed", "float64"):
        e.set_spins(S0)
        for c in range(SWEEPS // CHUNK):
            S = e.get_spins()
            row = {"sweeps": [c * CHUNK, (c + 1) * CHUNK]}
            for mode, name in ((("2", "stream"),) if path == "float64" else ()) + (("1", "plain"), ("0", "cold")):
                os.environ["ISB_SSF_MODE"] = mode
                e.set_spins(S)
                run(1, t0=c * CHUNK * N, fixed=path == "fixed")          # the field initialisation, not timed
                st = run(CHUNK * N - 1, t0=c * CHUNK * N + 1, fixed=path == "fixed")
                row[name + "_ms"] = st["kernel_ms"]
                row["acceptance"] = st["flips"] / (R * (CHUNK * N - 1))
                row["exact_fallbacks_" + name] = st["exact_fallbacks"]
            del os.environ["ISB_SSF_MODE"]
            prof[path].append(row)
            print(path, row, file=sys.stderr)
    res["profile"] = prof

    grid = []
    for thr_cold in args.thr.split(","):
        os.environ["ISB_SSF_COLD_THR"] = thr_cold
        ms = []
        for _ in range(args.reps):
            e.set_spins(S0)
            ms.append(run(SWEEPS * N)["kernel_ms"])
        grid.append({"thr_cold": float(thr_cold), "kernel_ms_median": float(np.median(ms))})
    del os.environ["ISB_SSF_COLD_THR"]
    res["thresholds"] = grid
    os.environ.pop("ISB_SSF_FIXED", None)

    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
