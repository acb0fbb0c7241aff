"""GPU tests of replica selection (isb_ens_select_replicas) and device-resident population annealing (isb_ssf_run_pa,
tempering.PopulationAnnealing).

The core check is a replay: every temperature step of isb_ssf_run_pa is by definition one traced isb_ssf_run of the
same steps, followed by one systematic resampling whose rule (weights, exact integer prefix sums, Philox offset, parent
search) is reproduced here in Python integers, applied with isb_ens_select_replicas.  Spins, traced E / M, families and
flip totals must be identical, lnQ equal to 1e-12.  The physics tests compare the free energy and the mean energy with
exact results (Kaufman's solution of the periodic lattice, enumeration of a small dense model), independently of the RNG."""
import numpy as np
import pytest

from oracle.oracle_np import philox4x32_10

pytestmark = pytest.mark.gpu

DOM_PA_RESAMPLE = 6
TWO32 = 1 << 32


def _lib():
    from isingmodel_jl_b200 import _lib
    return _lib


def _random_sparse(synth, n, deg, seed):
    """Symmetric sparse J with about `deg` neighbours per site and integer couplings."""
    import scipy.sparse as sp
    m = n * deg // 2
    i, j = synth.nodes(seed, n, m), synth.nodes(seed + 1, n, m)
    v = np.round(synth.gaussian(seed + 2, m) * 2.0)
    keep = i != j
    A = sp.coo_matrix((v[keep], (i[keep], j[keep])), shape=(n, n)).tocsr()
    A = sp.triu(A + A.T, 1)
    A = (A + A.T).tocsc()
    A.eliminate_zeros()
    return A


def _model(ctx, synth, kind):
    import scipy.sparse as sp
    L = _lib()
    if kind == "sk64_f64":
        return L.Model.dense(ctx, synth.sk_J(64, 11), synth.gaussian(12, 64) * 0.1, L.PREC_F64), 64
    if kind == "sk64_f32":
        return L.Model.dense(ctx, synth.sk_J(64, 13), None, L.PREC_F32), 64
    if kind == "dense1500":
        return L.Model.dense(ctx, synth.sk_J(1500, 14), None, L.PREC_F64), 1500
    if kind == "sparse300":
        return L.Model.sparse(ctx, _random_sparse(synth, 300, 6, 15), synth.gaussian(16, 300) * 0.25), 300
    if kind == "lattice32":
        return L.Model.sparse(ctx, sp.csc_matrix(synth.lattice_J(32)), np.zeros(1024)), 1024
    raise KeyError(kind)


def resample(E, T, Tn, K, seed, n_pop, near):
    """One resampling of the documented rule on the host, in Python integers.  Returns (parent [R] (global slots),
    lnQ [n_pop]).  Weights whose x * 2^32 lies within two ulps of an integer (where libm and the device exp could give
    different W) are appended to `near`."""
    R = E.size
    P = R // n_pop
    db = 1.0 / Tn - 1.0 / T
    parent, lnQ = np.zeros(R, dtype=np.int32), np.zeros(n_pop)
    for p in range(n_pop):
        a = -db * E[p * P:(p + 1) * P]
        amax = a.max()
        x = np.exp(a - amax)
        y = x * float(TWO32)
        dist = np.abs(y - np.round(y))
        for r in np.nonzero((dist < 2 * np.spacing(x) * TWO32) & (x != 1.0) & (x != 0.0))[0]:
            near.append((K, p, int(r), float(y[r])))
        W = [int(v) for v in np.floor(y)]
        C = np.cumsum(np.array(W, dtype=np.uint64))
        S = int(C[-1])
        U = int(philox4x32_10(np.uint32(K & 0xFFFFFFFF), np.uint32(K >> 32), np.uint32(p),
                              np.uint32(DOM_PA_RESAMPLE << 28), seed & 0xFFFFFFFF, seed >> 32)[0])
        t = np.array([((j << 32) + U) * S // (P << 32) for j in range(P)], dtype=np.uint64)
        parent[p * P:(p + 1) * P] = p * P + np.searchsorted(C, t, side="right")     # smallest r with C_r > t_j
        lnQ[p] = amax + np.log(x.sum() / P)
    return parent, lnQ


def replay(ens, rule, n_pop, T, T_next, spt, *, order, start, seed, step_offset, T_offset, family):
    """isb_ssf_run_pa rebuilt from isb_ssf_run calls, the host resampling and isb_ens_select_replicas."""
    R, n = ens.R, ens.nv
    nT = len(T)
    fam = np.array(family, dtype=np.int32)
    E, M = np.zeros((nT, R)), np.zeros((nT, R))
    lnQ, flips, near = [], np.zeros(R, dtype=np.int64), []
    for k in range(nT):
        out = ens.ssf_run(rule, spt, order=order, start=(start + k * spt) % n, seed=seed, step_offset=step_offset + k * spt,
                          T=np.array([T[k]]), steps_per_T=spt, trace_every=spt)
        E[k], M[k] = out["E"][0], out["M"][0]
        flips += out["flips"]
        if k < nT - 1 or T_next > 0:
            Tn = T[k + 1] if k < nT - 1 else T_next
            parent, q = resample(E[k], T[k], Tn, T_offset + k, seed, n_pop, near)
            ens.select_replicas(parent)
            fam = fam[parent]
            lnQ.append(q)
    return {"E": E, "M": M, "lnQ": np.array(lnQ).reshape(-1, n_pop), "family": fam, "flips": flips}, near


# (model, rule, order, populations, P, temperatures, steps per step, start, T_next as a factor of T0 (0: none))
CASES = [
    ("sk64_f64", 1, "seq", 2, 8, 6, 40, 5, 0.0),          # steps shorter than N
    ("sk64_f64", 2, "seq", 1, 16, 5, 64, 0, 0.5),         # equal to N, T_next given
    ("sk64_f64", 1, "seq", 4, 4, 5, 150, 63, 0.0),        # longer than N
    ("sk64_f32", 2, "seq", 2, 12, 6, 64, 3, 0.55),
    ("sk64_f64", 1, "random", 2, 8, 5, 100, 0, 0.0),
    ("dense1500", 1, "seq", 1, 8, 4, 1000, 17, 0.0),      # N > 1024: the neighbour-list path
    ("sparse300", 2, "seq", 2, 8, 5, 450, 11, 0.5),
    ("sparse300", 1, "seq", 4, 6, 5, 300, 0, 0.0),
    ("lattice32", 2, "seq", 2, 8, 5, 1024, 0, 0.0),
    ("lattice32", 2, "checkerboard", 2, 8, 4, 1500, 100, 0.6),
    ("lattice32", 1, "checkerboard", 1, 12, 5, 700, 0, 0.0),
]
# temperatures as factors of T0: cooling, with one heating step (db < 0) from the second to the third
SHAPE = np.array([1.0, 0.85, 0.95, 0.8, 0.7, 0.6])


@pytest.mark.parametrize("kind,rule,order,n_pop,P,nT,spt,start,tn", CASES)
def test_replay_parity(ctx, synth, kind, rule, order, n_pop, P, nT, spt, start, tn):
    L = _lib()
    o = {"seq": L.ORDER_SEQUENTIAL, "random": L.ORDER_RANDOM, "checkerboard": L.ORDER_CHECKERBOARD}[order]
    model, n = _model(ctx, synth, kind)
    R = n_pop * P
    T0 = {"sparse300": 3.0, "lattice32": 2.6}.get(kind, 0.8)
    T = T0 * SHAPE[:nT]
    T_next = T0 * tn
    S0 = synth.spins(21, R, n)
    fam0 = (np.arange(R, dtype=np.int32) * 7 + 3)          # arbitrary labels
    seed, off, toff = 0x1234ABCD5678, 977, 5
    a, b = L.Ensemble(model, R), L.Ensemble(model, R)
    a.set_spins(S0)
    b.set_spins(S0)
    got = a.ssf_run_pa(rule, n_pop, T, spt, T_next=T_next, order=o, start=start, seed=seed, step_offset=off, T_offset=toff,
                       family=fam0, want_M=True)
    want, near = replay(b, rule, n_pop, T, T_next, spt, order=o, start=start, seed=seed, step_offset=off, T_offset=toff,
                        family=fam0)
    print("near-integer weights:", near)
    assert not near
    assert np.array_equal(a.get_spins(), b.get_spins())
    assert np.array_equal(got["E"], want["E"]) and np.array_equal(got["M"], want["M"])
    assert np.array_equal(got["family"], want["family"])
    assert np.array_equal(got["flips"], want["flips"])
    assert got["lnQ"].shape == (nT - 1 + (T_next > 0), n_pop)
    assert np.allclose(got["lnQ"], want["lnQ"], rtol=1e-12, atol=1e-12)
    st = a.last_stats()
    assert st["flips"] == int(want["flips"].sum()) and st["kernel_ms"] > 0
    # the ensemble keeps a consistent state: a plain run continues both identically
    ra = a.ssf_run(rule, 2 * n, seed=3, T=np.array([T[-1]]), steps_per_T=2 * n, trace_every=n)
    rb = b.ssf_run(rule, 2 * n, seed=3, T=np.array([T[-1]]), steps_per_T=2 * n, trace_every=n)
    assert np.array_equal(a.get_spins(), b.get_spins()) and np.array_equal(ra["E"], rb["E"])


def test_replay_resamples(ctx, synth):
    """The replay cases above exercise real resampling: families die out."""
    L = _lib()
    model, n = _model(ctx, synth, "sk64_f64")
    e = L.Ensemble(model, 64)
    e.set_spins(synth.spins(23, 64, n))
    out = e.ssf_run_pa(1, 2, 0.8 * SHAPE, 64, seed=9, family=np.arange(64))
    assert all(len(np.unique(f)) < 32 for f in out["family"].reshape(2, 32))
    assert np.all(out["family"].reshape(2, 32) // 32 == np.arange(2)[:, None])   # populations stay apart


# ------------------------------------------------------------------ isb_ens_select_replicas
def _select_case(ctx, synth, kind, traced):
    """k steps, select_replicas(src) with repeats, m more steps against a control without the selection: slot j must
    continue exactly like the control's slot src[j] (shared fluctuations, sequential order)."""
    L = _lib()
    if kind == "dense":
        n = 96
        model = L.Model.dense(ctx, synth.sk_J(n, 81), synth.gaussian(82, n) * 0.3, L.PREC_F64)
    else:
        model, n = _model(ctx, synth, kind)
    R = 10
    src = np.array([3, 3, 0, 9, 9, 9, 1, 4, 2, 3], dtype=np.int32)
    S0 = synth.spins(83, R, n)
    k, mm = 7 * n + 13, 5 * n + 7
    fl = synth.logistic(84, (k + mm,))
    T = np.array([0.9 if kind != "lattice32" else 2.3])
    a, c = L.Ensemble(model, R), L.Ensemble(model, R)
    a.set_spins(S0)
    c.set_spins(S0)
    te = n if traced else 0
    kw = dict(fluct=fl[:k], T=T, steps_per_T=k, trace_every=te)
    a.ssf_run(1, k, **kw)
    c.ssf_run(1, k, **kw)
    a.select_replicas(src)
    kw = dict(fluct=fl[k:], T=T, steps_per_T=mm, trace_every=te, start=k % n)
    ra = a.ssf_run(1, mm, **kw)
    rc = c.ssf_run(1, mm, **kw)
    assert np.array_equal(a.get_spins(), c.get_spins()[src])
    if traced:
        assert np.array_equal(ra["E"], rc["E"][:, src]) and np.array_equal(ra["M"], rc["M"][:, src])
    assert np.array_equal(a.energy(), c.energy()[src])


@pytest.mark.parametrize("kind,traced", [("dense", True), ("dense", False), ("sparse300", True), ("lattice32", True),
                                         ("sk64_f32", True)])
def test_select_keeps_the_chain_state(ctx, synth, kind, traced):
    _select_case(ctx, synth, kind, traced)


def test_select_errors_leave_the_ensemble_unchanged(ctx, synth):
    L = _lib()
    n, R = 32, 6
    e = L.Ensemble(L.Model.dense(ctx, synth.sk_J(n, 91), None, L.PREC_F64), R)
    S0 = synth.spins(92, R, n)
    e.set_spins(S0)
    e.ssf_run(1, 3 * n, seed=1, T=np.array([1.0]), steps_per_T=3 * n, trace_every=n)
    ref = e.clone()
    ref.set_spins(e.get_spins())
    for bad, code in ((np.array([0, 1, 2, 3, 4, 6]), L.ERR_ARG), (np.array([0, 1, -1, 3, 4, 5]), L.ERR_ARG),
                      (np.arange(R - 1), L.ERR_SIZE), (np.arange(R + 1), L.ERR_SIZE)):
        with pytest.raises(L.IsbError) as ei:
            e.select_replicas(bad)
        assert ei.value.code == code
    W, hv, hb = synth.bipartite_W(8, 4, 93)
    bip = L.Ensemble(L.Model.bipartite(ctx, W, hv, hb), R)
    with pytest.raises(L.IsbError) as ei:
        bip.select_replicas(np.arange(R))
    assert ei.value.code == L.ERR_STATE
    assert np.array_equal(e.get_spins(), ref.get_spins())
    ra = e.ssf_run(1, 2 * n, seed=2, T=np.array([1.0]), steps_per_T=2 * n, trace_every=n)
    rb = ref.ssf_run(1, 2 * n, seed=2, T=np.array([1.0]), steps_per_T=2 * n, trace_every=n)
    assert np.array_equal(e.get_spins(), ref.get_spins()) and np.allclose(ra["E"], rb["E"], rtol=1e-12)


# ------------------------------------------------------------------ identity and continuation
def test_equal_temperatures_are_the_identity(ctx, synth):
    L = _lib()
    model, n = _model(ctx, synth, "sk64_f64")
    R, spt, nT = 24, 2 * n, 5
    S0 = synth.spins(101, R, n)
    a, b = L.Ensemble(model, R), L.Ensemble(model, R)
    a.set_spins(S0)
    b.set_spins(S0)
    fam = np.arange(R, dtype=np.int32)
    got = a.ssf_run_pa(1, 3, np.full(nT, 0.7), spt, T_next=0.7, start=4, seed=5, step_offset=11, family=fam)
    one = b.ssf_run(1, nT * spt, start=4, seed=5, step_offset=11, T=np.array([0.7]), steps_per_T=nT * spt,
                    trace_every=spt)
    assert np.array_equal(got["family"], fam)
    assert np.array_equal(a.get_spins(), b.get_spins())
    assert np.array_equal(got["flips"], one["flips"])
    assert np.allclose(got["E"], one["E"], rtol=1e-12, atol=1e-12)
    assert np.all(got["lnQ"] == 0.0)


def test_two_calls_equal_one(ctx, synth):
    L = _lib()
    model, n = _model(ctx, synth, "sk64_f64")
    R, spt, a_, b_ = 32, 48, 4, 9
    T = 1.2 * np.geomspace(1.0, 0.4, b_)
    S0 = synth.spins(111, R, n)
    x, y = L.Ensemble(model, R), L.Ensemble(model, R)
    x.set_spins(S0)
    y.set_spins(S0)
    fam = np.arange(R, dtype=np.int32)
    one = x.ssf_run_pa(2, 2, T, spt, start=9, seed=7, step_offset=100, T_offset=3, family=fam, want_M=True)
    p1 = y.ssf_run_pa(2, 2, T[:a_], spt, T_next=T[a_], start=9, seed=7, step_offset=100, T_offset=3, family=fam,
                      want_M=True)
    p2 = y.ssf_run_pa(2, 2, T[a_:], spt, start=(9 + a_ * spt) % n, seed=7, step_offset=100 + a_ * spt, T_offset=3 + a_,
                      family=p1["family"], want_M=True)
    assert np.array_equal(x.get_spins(), y.get_spins())
    for key in ("E", "M", "lnQ"):
        assert np.array_equal(one[key], np.concatenate([p1[key], p2[key]])), key
    assert np.array_equal(one["family"], p2["family"])
    assert np.array_equal(one["flips"], p1["flips"] + p2["flips"])


def test_class_continues_across_runs(pkg, ctx, synth):
    """PopulationAnnealing: run() calls continue one anneal (family, lnZ, offsets) and mark the host spins stale."""
    n, R = 64, 48
    J = synth.sk_J(n, 121)
    T = np.geomspace(1.5, 0.5, 8)
    res = []
    for split in ((8,), (3, 5)):
        ss = pkg.SpinSystems.SpinSystem(synth.spins(122, R, n), J, np.zeros(n))
        pa = pkg.tempering.PopulationAnnealing(pkg.SingleSpinFlip.GlauberDynamics(ss, 1.0), populations=3, seed=4)
        Es, i = [], 0
        for s in split:
            nxt = T[i + s] if i + s < len(T) else None
            Es.append(pa.run(T[i:i + s], sweeps=2, next_temperature=nxt))
            i += s
        res.append((pa, ss, np.concatenate(Es)))
    (p1, s1, E1), (p2, s2, E2) = res
    assert E1.shape == (8, 3, 16) and np.array_equal(E1, E2)
    assert np.array_equal(s1.spinConfiguration, s2.spinConfiguration)
    assert np.array_equal(p1.family, p2.family) and np.allclose(p1.lnZ, p2.lnZ, rtol=1e-12, atol=1e-12)
    assert p1.offset == p2.offset == 8 * 2 * n and p1.step == p2.step == 8 and p1.temperature == T[-1]
    st = p1.family_statistics()
    assert np.all(st["families"] >= 1) and np.all(st["families"] <= 16)
    assert np.all(st["rho_t"] >= 1.0) and np.all(st["entropy"] <= np.log(16) + 1e-12)
    # the energies it reports are those of the spins it leaves (no resampling after the last temperature)
    Ecur = np.asarray(pkg.SpinSystems.calcEnergy(p1.ua)).reshape(-1)
    assert np.allclose(Ecur, E1[-1].reshape(-1), rtol=1e-9, atol=1e-9)
    with pytest.raises(ValueError):
        p1.run([0.9])                     # the populations are at T[-1], not 0.9


# ------------------------------------------------------------------ physics, independent of the RNG
# Tolerance rule: the populations are independent estimates, so each quantity is compared as
#   |mean over populations - exact| < 5 * (standard deviation over populations, ddof = 1) / sqrt(populations)
# plus a floor of 1e-3 of the exact value for E (and 1e-9 absolute for ln Z), which only matters where the spread is tiny.
def _check(est, exact, floor, what):
    m, se = est.mean(0), est.std(0, ddof=1) / np.sqrt(est.shape[0])
    bad = np.abs(m - exact) >= 5 * se + floor
    assert not bad.any(), (what, np.nonzero(bad)[0], m[bad], np.asarray(exact)[bad], se[bad])


def test_lattice_free_energy_and_energy_match_kaufman(pkg, ctx, synth):
    import scipy.sparse as sp
    from exact_ising import ln_partition, mean_energy
    Ls, npop, P = 32, 8, 2048
    N, R = Ls * Ls, npop * P
    ss = pkg.SpinSystems.SpinSystem(synth.spins(131, R, N), sp.csc_matrix(synth.lattice_J(Ls)), np.zeros(N))
    pa = pkg.tempering.PopulationAnnealing(pkg.SingleSpinFlip.MetropolisMethod(ss, 1.0), populations=npop, seed=13)
    T = np.geomspace(5.0, 2.3, 60)
    pa.run(np.full(10, T[0]), sweeps=2)                 # equilibrate at T[0] (equal temperatures: no resampling)
    E = pa.run(T, sweeps=2)                             # [nT][populations][P]
    lnZ = pa.lnZ_run - pa.lnZ_run[0]                    # ln Z(T_k) / Z(T_0) per population
    exact = np.array([ln_partition(Ls, Ls, 1.0 / t) - ln_partition(Ls, Ls, 1.0 / T[0]) for t in T])
    ks = np.arange(5, len(T), 5)
    _check(lnZ[ks].T, exact[ks], 1e-9, "lnZ")
    exE = np.array([mean_energy(Ls, t) for t in T[ks]])
    _check(E.mean(2)[ks].T, exE, 1e-3 * np.abs(exE), "E")
    assert np.all(pa.family_statistics()["families"] > 1)


def test_dense_free_energy_and_energy_match_enumeration(pkg, ctx, synth):
    n, npop, P = 12, 8, 1024
    J, h = synth.sk_J(n, 141) * 2.0, synth.gaussian(142, n) * 0.3
    ss = pkg.SpinSystems.SpinSystem(synth.spins(143, npop * P, n), J, h)
    pa = pkg.tempering.PopulationAnnealing(pkg.SingleSpinFlip.GlauberDynamics(ss, 1.0), populations=npop, seed=14)
    T = np.geomspace(3.0, 0.6, 40)
    pa.run(np.full(20, T[0]))
    E = pa.run(T)
    states = 1 - 2 * ((np.arange(1 << n)[:, None] >> np.arange(n)) & 1)
    Es = -0.5 * np.einsum("ki,ij,kj->k", states, J, states) - states @ h

    def lnZ(t):
        a = -Es / t
        return a.max() + np.log(np.exp(a - a.max()).sum())

    def meanE(t):
        w = np.exp(-(Es - Es.min()) / t)
        return float((Es * w).sum() / w.sum())

    ks = np.arange(4, len(T), 4)
    _check((pa.lnZ_run - pa.lnZ_run[0])[ks].T, np.array([lnZ(T[k]) - lnZ(T[0]) for k in ks]), 1e-9, "lnZ")
    ex = np.array([meanE(T[k]) for k in ks])
    _check(E.mean(2)[ks].T, ex, 1e-3 * np.abs(ex), "E")


# ------------------------------------------------------------------ full size
def test_full_size_c2(ctx, synth):
    """C2's model (SK N = 1024, Gaussian J), 4096 replicas in one population, the first temperature steps of C2's schedule
    as population annealing runs it (2.0 -> 0.05 in 200 steps) on the register-kernel path: the replay holds, lnQ is
    finite and more than one family survives."""
    L = _lib()
    n, R = 1024, 4096
    model = L.Model.dense(ctx, synth.sk_J(n, 2), np.zeros(n), L.PREC_F64)
    sched = np.geomspace(2.0, 0.05, 200)
    T = sched[:4]
    S0 = synth.spins(3, R, n)
    a, b = L.Ensemble(model, R), L.Ensemble(model, R)
    a.set_spins(S0)
    b.set_spins(S0)
    fam = np.arange(R, dtype=np.int32)
    got = a.ssf_run_pa(1, 1, T, n, T_next=sched[4], seed=12345, family=fam, want_M=True)
    want, near = replay(b, 1, 1, T, sched[4], n, order=L.ORDER_SEQUENTIAL, start=0, seed=12345, step_offset=0,
                        T_offset=0, family=fam)
    print("near-integer weights:", near)
    assert not near
    assert np.array_equal(a.get_spins(), b.get_spins())
    assert np.array_equal(got["E"], want["E"]) and np.array_equal(got["M"], want["M"])
    assert np.array_equal(got["family"], want["family"]) and np.array_equal(got["flips"], want["flips"])
    assert np.all(np.isfinite(got["lnQ"])) and np.allclose(got["lnQ"], want["lnQ"], rtol=1e-12, atol=1e-12)
    assert 1 < len(np.unique(got["family"])) < R


# ------------------------------------------------------------------ validation
def test_errors_leave_the_ensemble_unchanged(ctx, synth):
    L = _lib()
    n, R = 32, 12
    model = L.Model.dense(ctx, synth.sk_J(n, 151), None, L.PREC_F64)
    e = L.Ensemble(model, R)
    S0 = synth.spins(152, R, n)
    e.set_spins(S0)
    fam = np.arange(R, dtype=np.int32)
    T = np.array([1.0, 0.8, 0.6])

    def expect(code, *args, ens=e, **kw):
        kw.setdefault("family", fam)
        before = None if kw["family"] is None else np.array(kw["family"], copy=True)
        with pytest.raises(L.IsbError) as ei:
            ens.ssf_run_pa(*args, **kw)
        assert ei.value.code == code and ei.value.message, (code, ei.value)
        if before is not None:
            assert np.array_equal(kw["family"], before)

    W, hv, hb = synth.bipartite_W(8, 4, 153)
    expect(L.ERR_STATE, 1, 2, T, n, ens=L.Ensemble(L.Model.bipartite(ctx, W, hv, hb), R))
    expect(L.ERR_ARG, L.RULE_HOPFIELD, 2, T, n)
    expect(L.ERR_ARG, 1, 2, T, n, order=L.ORDER_LIST)
    expect(L.ERR_UNSUPPORTED, 1, 2, T, n, order=L.ORDER_CHECKERBOARD)      # a dense model is not a lattice
    expect(L.ERR_SIZE, 1, 5, T, n)
    expect(L.ERR_ARG, 1, 0, T, n)
    expect(L.ERR_ARG, 1, 2, np.array([1.0, 0.0, 0.6]), n)
    expect(L.ERR_ARG, 1, 2, np.array([1.0, -0.8, 0.6]), n)
    expect(L.ERR_NONFINITE, 1, 2, np.array([1.0, np.nan, 0.6]), n)
    expect(L.ERR_NONFINITE, 1, 2, np.array([1.0, np.inf, 0.6]), n)
    expect(L.ERR_ARG, 1, 2, T, n, T_next=-0.5)
    expect(L.ERR_NONFINITE, 1, 2, T, n, T_next=np.inf)
    expect(L.ERR_ARG, 1, 2, T, 0)
    expect(L.ERR_ARG, 1, 2, T, n, start=n)
    e.set_temperature_scale(np.linspace(0.5, 1.5, R))
    expect(L.ERR_STATE, 1, 2, T, n)
    e.set_temperature_scale(None)
    big = L.Ensemble(L.Model.dense(ctx, synth.sk_J(32, 154), None, L.PREC_F64), (1 << 20) + 1)
    expect(L.ERR_UNSUPPORTED, 1, 1, T, n, ens=big, family=None)             # P = 2^20 + 1
    del big
    # nT = 0 is a no-op
    out = e.ssf_run_pa(1, 2, np.zeros(0), n, family=fam)
    assert np.array_equal(out["family"], fam) and not out["flips"].any() and out["lnQ"].shape == (0, 2)
    # nothing moved
    assert np.array_equal(e.get_spins(), S0)
