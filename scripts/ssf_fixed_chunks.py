"""Chunk times of one build of the fixed-point dense sweep kernels on the C2 anneal (SK N = 1024, 4096 replicas,
Glauber, 1000 sweeps of bench.py's geometric schedule, Philox noise), for comparing builds: run it once per library
with ISING_B200_LIB pointing at each.  The chunks are measured as in ssf_fixed_ab.py (each 50-sweep chunk started from
the anneal's state with the kernel forced by ISB_SSF_MODE, the field initialisation not timed), best of two, and the
anneal is carried forward on the plain kernel.  Prints one JSON line (and writes it to --out).

    ISING_B200_LIB=$PWD/scratch_ab/lib_x.so python scripts/ssf_fixed_chunks.py --tag x --plain 0,4,7,8 --cold 8

With --libs, the builds are alternated within one call: each round runs this script once per library, in a
subprocess, and the output lists every run and, per build and chunk, the best time over the rounds.

    python scripts/ssf_fixed_chunks.py --libs a=scratch_ab/lib_a.so,b=scratch_ab/lib_b.so --rounds 2 --plain all"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

N, R, SWEEPS, CHUNK = 1024, 4096, 1000, 50


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tag", default="build")
    ap.add_argument("--plain", default="0,4", help="chunks timed on the plain kernel")
    ap.add_argument("--cold", default="", help="chunks timed on the cold kernel")
    ap.add_argument("--anneals", type=int, default=2, help="whole anneals timed (after one untimed)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--libs", default=None, help="tag=path,...: alternate these builds, one subprocess per run")
    ap.add_argument("--rounds", type=int, default=2, help="with --libs: runs of each build")
    args = ap.parse_args()
    everything = ",".join(str(c) for c in range(SWEEPS // CHUNK))
    args.plain, args.cold = (everything if v == "all" else v for v in (args.plain, args.cold))
    if args.libs:
        return alternate(args)
    import bench
    from isingmodel_jl_b200 import _lib as L, synth
    from ssf_fixed_ab import card
    plain = [int(c) for c in args.plain.split(",") if c]
    cold = [int(c) for c in args.cold.split(",") if c]
    J, h, T = bench.workload(SWEEPS)
    S0 = synth.spins(bench.SEED_S, R, N)
    ctx = L.context(0)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)

    def run(nsteps, t0=0):
        e.ssf_run(L.RULE_GLAUBER, nsteps, start=t0 % N, seed=12345, step_offset=t0, T=T[t0 // N:], steps_per_T=N)
        return e.last_stats()

    res = {"tag": args.tag, "lib": L.LIB_PATH, "card": card(), "anneal": [], "chunks": {}}
    for rep in range(args.anneals + 1):
        e.set_spins(S0)
        st = run(SWEEPS * N)
        if rep:
            res["anneal"].append({k: st[k] for k in ("kernel_ms", "flips", "exact_fallbacks")})
    e.set_spins(S0)
    for c in range(max(plain + cold) + 1):
        S = e.get_spins()
        row = {}
        for mode, name, which in (("1", "plain", plain), ("0", "cold", cold)):
            if c not in which:
                continue
            os.environ["ISB_SSF_MODE"] = mode
            ms = []
            for _ in range(2):
                e.set_spins(S)
                run(1, t0=c * CHUNK * N)   # the field initialisation, not timed
                st = run(CHUNK * N - 1, t0=c * CHUNK * N + 1)
                ms.append(st["kernel_ms"])
            row[name + "_ms"] = min(ms)
            row["acceptance"] = st["flips"] / (R * (CHUNK * N - 1))
        os.environ["ISB_SSF_MODE"] = "1"   # carry the anneal forward
        e.set_spins(S)
        run(1, t0=c * CHUNK * N)
        run(CHUNK * N - 1, t0=c * CHUNK * N + 1)
        del os.environ["ISB_SSF_MODE"]
        if row:
            res["chunks"][c] = row
    write(res, args.out)


def write(res, out):
    txt = json.dumps(res)
    print(txt)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(txt + "\n")


def alternate(args):
    libs = [kv.split("=", 1) for kv in args.libs.split(",")]
    runs = []
    for rnd in range(args.rounds):
        for tag, path in libs:
            cmd = [sys.executable, os.path.abspath(__file__), "--tag", tag, "--plain", args.plain, "--cold", args.cold,
                   "--anneals", str(args.anneals)]
            env = dict(os.environ, ISING_B200_LIB=os.path.abspath(path))
            out = subprocess.run(cmd, env=env, check=True, capture_output=True, text=True).stdout
            run = json.loads(out.strip().splitlines()[-1])
            run["round"] = rnd
            runs.append(run)
            print(json.dumps({k: run[k] for k in ("tag", "round", "anneal")}), file=sys.stderr)
    best = {}
    for run in runs:
        b = best.setdefault(run["tag"], {"anneal_ms": [], "chunks": {}})
        b["anneal_ms"] += [a["kernel_ms"] for a in run["anneal"]]
        for c, row in run["chunks"].items():
            bc = b["chunks"].setdefault(c, {})
            for k, v in row.items():
                bc[k] = min(bc.get(k, v), v) if k.endswith("_ms") else v
    write({"card": runs[0]["card"], "runs": runs, "best": best}, args.out)


if __name__ == "__main__":
    main()
