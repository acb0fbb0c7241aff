"""Swendsen-Wang sweeps (isb_sw_run) against the Metropolis single-spin sweep on the same ensembles.  Prints one JSON
document (and writes it to --out).

  (a) sweep time: device time per sweep (isb_ens_last_stats over --sweeps sweeps, best of --reps calls) of the SW kernel
      and of a sequential Metropolis isb_ssf_run of the same ensemble, for the ferromagnetic torus at T_c with L = 32
      (R = 4096), 64 (R = 1024), 128 (R = 256) and a 64 x 64 +-J torus at T = 1;
  (b) decorrelation at T_c, L = 32 and 64: integrated autocorrelation times (Sokal's window, c = 6) of E and M^2 from
      every-sweep traces of equilibrated replicas (both dynamics start from the same SW-equilibrated spins), the
      autocorrelation function averaged over the replicas;
  (c) net rate: independent samples per device-second, R / (2 tau_int(M^2) * device time per sweep of the ensemble).
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

TC = 2.0 / np.log(1.0 + np.sqrt(2.0))


def card():
    info = {}
    try:   # read-only query
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except (OSError, subprocess.TimeoutExpired) as exc:
        info["nvidia_smi"] = f"unavailable: {exc}"
    return info


def torus(L, pm_seed=None):
    import scipy.sparse as sp
    from isingmodel_jl_b200 import synth
    J = sp.csc_matrix(synth.lattice_J(L))
    if pm_seed is None:
        return J
    A = sp.triu(J, 1).tocoo()
    v = np.where(synth.uniform01(pm_seed, A.nnz) < 0.5, -1.0, 1.0)
    U = sp.coo_matrix((v, (A.row, A.col)), shape=A.shape)
    return (U + U.T).tocsc()


def ensemble(J, R, seed):
    from isingmodel_jl_b200 import _lib
    n = J.shape[0]
    ens = _lib.Ensemble(_lib.Model.sparse(_lib.context(0), J, np.zeros(n)), R)
    ens.set_spins(np.where(np.random.default_rng(seed).random((R, n)) < 0.5, -1, 1).astype(np.int8))
    return ens


def sweep_times(J, R, T, sweeps, reps):
    from isingmodel_jl_b200 import _lib
    n = J.shape[0]
    ens = ensemble(J, R, 1)
    ens.sw_run(20, T, sweeps_per_T=20, seed=1)          # warm-up (and the one-time bond list)
    sw, me = [], []
    off = 20
    for _ in range(reps):
        ens.sw_run(sweeps, T, sweeps_per_T=sweeps, seed=1, sweep_offset=off)
        off += sweeps
        sw.append(ens.last_stats()["kernel_ms"] / sweeps)
        ens.ssf_run(_lib.RULE_METROPOLIS, sweeps * n, T=[T], steps_per_T=sweeps * n, seed=2, step_offset=off * n)
        me.append(ens.last_stats()["kernel_ms"] / sweeps)
    return {"sw_ms_per_sweep": min(sw), "metropolis_ms_per_sweep": min(me), "sw_all": sw, "metropolis_all": me,
            "sw_over_metropolis": min(sw) / min(me)}


def tau_int(x):
    """x: [t][R] series of R independent replicas -> Sokal-window integrated autocorrelation time (c = 6)."""
    x = x - x.mean(axis=0)
    t = x.shape[0]
    acf = np.zeros(t)
    for c in range(0, x.shape[1], 32):          # (in column blocks: the transforms of a long series are large)
        f = np.fft.rfft(x[:, c:c + 32], n=2 * t, axis=0)
        acf += np.fft.irfft(f * np.conj(f), axis=0)[:t].sum(axis=1)
    acf /= acf[0]
    tau = 0.5
    for w in range(1, t):
        tau += acf[w]
        if w >= 6.0 * tau:
            return float(tau), w
    return float(tau), t


def decorrelation(L, R, sw_sweeps, me_sweeps):
    from isingmodel_jl_b200 import _lib
    J = torus(L)
    n = L * L
    ens = ensemble(J, R, 3)
    ens.sw_run(1000, TC, sweeps_per_T=1000, seed=3)                   # equilibrate
    S = ens.get_spins()
    out = {}
    o = ens.sw_run(sw_sweeps, TC, sweeps_per_T=sw_sweeps, trace_every=1, seed=3, sweep_offset=1000)
    sw_ms = ens.last_stats()["kernel_ms"] / sw_sweeps
    for name, x in (("E", o["E"]), ("M2", o["M"] ** 2)):
        tau, w = tau_int(x)
        out[f"sw_tau_{name}"], out[f"sw_window_{name}"] = tau, w
    me = ensemble(J, R, 4)
    me.set_spins(S)
    chunk = max(1, min(me_sweeps, (1 << 28) // (R * 8)))
    Es, Ms, me_ms = [], [], 0.0
    done = 0
    while done < me_sweeps:
        c = min(chunk, me_sweeps - done)
        r = me.ssf_run(_lib.RULE_METROPOLIS, c * n, T=[TC], steps_per_T=c * n, seed=5, step_offset=done * n, trace_every=n)
        me_ms += me.last_stats()["kernel_ms"]
        Es.append(r["E"])
        Ms.append(r["M"])
        done += c
    me_ms /= me_sweeps
    for name, x in (("E", np.concatenate(Es)), ("M2", np.concatenate(Ms) ** 2)):
        tau, w = tau_int(x)
        out[f"metropolis_tau_{name}"], out[f"metropolis_window_{name}"] = tau, w
    out.update({"L": L, "replicas": R, "sw_sweeps": sw_sweeps, "metropolis_sweeps": me_sweeps,
                "sw_ms_per_sweep_traced": sw_ms, "metropolis_ms_per_sweep_traced": me_ms})
    # net rate: independent samples (of M^2) per device-second of the ensemble
    out["sw_samples_per_s"] = R / (2.0 * out["sw_tau_M2"] * sw_ms * 1e-3)
    out["metropolis_samples_per_s"] = R / (2.0 * out["metropolis_tau_M2"] * me_ms * 1e-3)
    out["sw_over_metropolis_samples"] = out["sw_samples_per_s"] / out["metropolis_samples_per_s"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sw-series", type=int, default=4000)
    ap.add_argument("--metropolis-series", type=str, default="32:20000,64:40000")
    ap.add_argument("--decorrelation-replicas", type=int, default=512)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    doc = {"card": card(), "args": vars(a), "T_c": TC, "sweep_time": {}, "decorrelation": {}}
    for name, L, R, T, pm in (("ferro_L32_R4096_Tc", 32, 4096, TC, None), ("ferro_L64_R1024_Tc", 64, 1024, TC, None),
                              ("ferro_L128_R256_Tc", 128, 256, TC, None), ("pmJ_L64_R1024_T1", 64, 1024, 1.0, 11)):
        doc["sweep_time"][name] = {"L": L, "replicas": R, "T": T, **sweep_times(torus(L, pm), R, T, a.sweeps, a.reps)}
        print(name, json.dumps(doc["sweep_time"][name]), flush=True)
    for item in a.metropolis_series.split(","):
        L, ms = (int(v) for v in item.split(":"))
        doc["decorrelation"][f"L{L}"] = decorrelation(L, a.decorrelation_replicas, a.sw_series, ms)
        print(f"L{L}", json.dumps(doc["decorrelation"][f"L{L}"]), flush=True)
    txt = json.dumps(doc, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()
