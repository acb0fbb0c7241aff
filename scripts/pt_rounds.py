"""Parallel tempering at one sweep per round: the host-driven tempering.ParallelTempering against the device-resident
tempering.DeviceParallelTempering (isb_ssf_run_pt), on C2's model (SK N = 1024, Glauber) and C1's (32 x 32 torus,
Metropolis), 32 levels x 128 ladders = 4096 replicas each.  Prints one JSON document (and writes it to --out).

Per model: rounds/s and spin updates/s of both classes (wall clock around whole run() calls, both of which end in a
device synchronisation, after warm-up rounds), the device time of the sweeps alone (isb_ens_last_stats of plain
isb_ssf_run calls of one round's steps each, and of one call of all the rounds' steps), the device time of the
isb_ssf_run_pt call, and the kernel totals of a separate torch.profiler run of the device class."""
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


def system(kind, R):
    import scipy.sparse as sp
    from isingmodel_jl_b200 import SingleSpinFlip, SpinSystems, synth
    if kind == "c2":
        N = 1024
        ss = SpinSystems.SpinSystem(synth.spins(3, R, N), synth.sk_J(N, 2), np.zeros(N))
        return ss, SingleSpinFlip.GlauberDynamics(ss, 1.0), np.geomspace(0.4, 2.0, 32)
    N = 1024
    ss = SpinSystems.SpinSystem(synth.spins(3, R, N), sp.csc_matrix(synth.lattice_J(32)), np.zeros(N))
    return ss, SingleSpinFlip.MetropolisMethod(ss, 1.0), np.linspace(1.6, 3.2, 32)


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t


def measure(kind, args):
    import torch
    from isingmodel_jl_b200 import _lib as L, tempering
    R, N = 4096, 1024
    res = {"model": {"c2": "SK N=1024 dense Gaussian J, Glauber", "c1": "32x32 periodic ferromagnet (sparse J), Metropolis"}[kind],
           "levels": 32, "ladders": 128, "replicas": R, "sweeps_per_round": 1}

    ss, ua, levels = system(kind, R)
    host = tempering.ParallelTempering(ua, levels, seed=1)
    host.run(args.warmup)
    _, dt = timed(lambda: host.run(args.host_rounds))
    res["host_class"] = {"rounds": args.host_rounds, "seconds": dt, "rounds_per_s": args.host_rounds / dt,
                         "updates_per_s": args.host_rounds * N * R / dt}

    ss, ua, levels = system(kind, R)
    dev = tempering.DeviceParallelTempering(ua, levels, seed=1)
    dev.run(args.warmup)
    ens = ss._ensemble()
    _, dt = timed(lambda: dev.run(args.rounds))
    st = ens.last_stats()
    res["device_class"] = {"rounds": args.rounds, "seconds": dt, "rounds_per_s": args.rounds / dt,
                           "updates_per_s": args.rounds * N * R / dt, "pt_call_device_ms": st["kernel_ms"],
                           "launches": st["launches"]}
    _, dt = timed(lambda: dev.run(args.rounds, overlaps=True))
    st = ens.last_stats()
    res["device_class_with_overlaps"] = {"rounds": args.rounds, "seconds": dt, "rounds_per_s": args.rounds / dt,
                                         "pt_call_device_ms": st["kernel_ms"], "launches": st["launches"]}
    res["speedup_rounds_per_s"] = res["device_class"]["rounds_per_s"] / res["host_class"]["rounds_per_s"]

    # the sweeps alone, on the same ensemble and ladder state: one isb_ssf_run per round, and all rounds in one call
    ens.set_temperature_scale(ua.temperatureScale)
    o = L.ORDER_SEQUENTIAL
    ms = 0.0
    for k in range(args.rounds):
        ens.ssf_run(ua._rule, N, order=o, seed=9, step_offset=k * N, T=np.array([1.0]), steps_per_T=N, trace_every=N,
                    want_M=False)
        ms += ens.last_stats()["kernel_ms"]
    res["sweeps_alone"] = {"per_round_calls_device_ms": ms,
                           "per_round_device_us": 1e3 * ms / args.rounds}
    ens.ssf_run(ua._rule, N * args.rounds, order=o, seed=9, T=np.array([1.0]), steps_per_T=N * args.rounds,
                trace_every=N, want_M=False)
    res["sweeps_alone"]["one_call_device_ms"] = ens.last_stats()["kernel_ms"]
    pt = res["device_class"]["pt_call_device_ms"]
    res["pt_device_ms_over_sweeps_alone"] = pt / ms
    res["pt_with_overlaps_device_ms_over_sweeps_alone"] = res["device_class_with_overlaps"]["pt_call_device_ms"] / ms

    # kernel totals of the device class (a separate, profiled run)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dev.run(args.profile_rounds, overlaps=True)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        if us > 0:
            kern[ev.key[:90]] = {"calls": ev.count, "total_us": us}
    res["profiled_kernels"] = {"rounds": args.profile_rounds, "kernels": kern}
    ens.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2000)
    ap.add_argument("--host-rounds", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--profile-rounds", type=int, default=100)
    ap.add_argument("--models", default="c2,c1")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("pt_rounds.py measures on a CUDA device; none is visible")
    doc = {"card": card(), "args": vars(args), "results": {}}
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
