"""GPU parity tests of the sparse-coupling single-spin path (isb_model_sparse) against the CPU oracle (which
takes the same J densified): bit-exact spins / flips / magnetisation, energies to 1e-9."""
import numpy as np
import pytest

from cases import golden_J, nodes_of
from conftest import load_golden

pytestmark = pytest.mark.gpu


def _close(a, b):
    return np.all(np.abs(a - b) <= 1e-9 * np.maximum(1.0, np.abs(b)))


def _lib():
    from isingmodel_jl_b200 import _lib
    return _lib


def _random_sparse(synth, n, deg, seed, integer):
    """Symmetric sparse J with about `deg` neighbours per site."""
    import scipy.sparse as sp
    m = n * deg // 2
    i = synth.nodes(seed, n, m)
    j = synth.nodes(seed + 1, n, m)
    v = synth.gaussian(seed + 2, m)
    if integer:
        v = np.round(v * 2.0)
    keep = i != j
    A = sp.coo_matrix((v[keep], (i[keep], j[keep])), shape=(n, n)).tocsr()
    A = sp.triu(A + A.T, 1)
    A = (A + A.T).tocsc()
    A.eliminate_zeros()
    return A


@pytest.mark.parametrize("name", ["ssf_2spin_glauber", "ssf_3x3_metropolis", "ssf_c1_32x32_metropolis", "ssf_sk64_glauber",
                                  "ssf_sk64_hopfield"])
def test_sparse_golden(ctx, synth, name):
    import scipy.sparse as sp
    L = _lib()
    g = load_golden(name)
    J = golden_J(name, g, synth)
    m = L.Model.sparse(ctx, sp.csc_matrix(J), g["h"])
    e = L.Ensemble(m, 1)
    e.set_spins(g["s0"][None, :])
    out = e.ssf_run(int(g["rule"]), int(g["nsteps"]), nodes=nodes_of(g), fluct=g["fluct"], T=g["T"],
                    steps_per_T=int(g["steps_per_T"]), trace_every=int(g["trace_every"]))
    assert np.array_equal(e.get_spins()[0], g["s_final"])
    assert int(out["flips"][0]) == int(g["flips"])
    assert np.array_equal(out["M"][:, 0], g["M"])
    assert _close(out["E"][:, 0], g["E"]) and _close(e.energy()[0], g["E"][-1])


CASES = [(50, 4, 1, "seq", 7, 50 * 9 + 3, True), (300, 6, 2, "list", 33, 2500, True), (1024, 4, 2, "seq", 200, 1024 * 3, False),
         (2000, 8, 1, "seq", 64, 2000 * 2 + 11, False), (5000, 3, 0, "seq", 9, 5000, True), (777, 10, 1, "list", 50, 3000, False)]


@pytest.mark.parametrize("n,deg,rule,order,R,nsteps,integer", CASES)
def test_sparse_batched_bit_exact(ctx, orc, synth, n, deg, rule, order, R, nsteps, integer):
    L = _lib()
    A = _random_sparse(synth, n, deg, 40 + n, integer)
    J = A.toarray()
    h = synth.gaussian(5, n) * 0.3
    S0 = synth.spins(6, R, n)
    nodes = synth.nodes(7, n, nsteps) if order == "list" else None
    fl = synth.logistic(8, (R, nsteps)) if rule == 1 else (synth.exponential(8, (R, nsteps)) if rule == 2 else None)
    T = synth.geometric_schedule(2.0, 0.2, 5)
    spT = (nsteps + 4) // 5
    e = L.Ensemble(L.Model.sparse(ctx, A, h), R)
    e.set_spins(S0)
    tr = max(1, nsteps // 2)
    out = e.ssf_run(rule, nsteps, nodes=nodes, start=n // 2 if order == "seq" else 0, fluct=fl, fluct_per_replica=True,
                    T=T, steps_per_T=spT, trace_every=tr)
    S = e.get_spins()
    for r in range(min(R, 12)):
        s, flips, E, M = orc.ssf_run(rule, J, h, S0[r], nsteps, nodes=nodes, start=n // 2 if order == "seq" else 0,
                                     fluct=None if fl is None else fl[r], T=T, steps_per_T=spT, trace_every=tr)
        assert np.array_equal(s, S[r]) and flips == out["flips"][r]
        assert np.array_equal(M, out["M"][:, r]) and _close(out["E"][:, r], E)
    Eg = e.energy()
    assert _close(Eg[:4], np.array([orc.energy(J, h, S[r]) for r in range(4)]))
    F = e.local_field()
    assert np.array_equal(F[0], orc.local_field(J, h, S[0]))


def test_sparse_equals_dense_path(ctx, synth):
    """The same lattice through the sparse and the dense kernels, Philox noise: identical trajectories."""
    import scipy.sparse as sp
    L = _lib()
    J = synth.lattice_J(32)
    S0 = synth.spins(1, 64, 1024)
    T = np.full(8, 2.269)
    res = []
    for model in (L.Model.dense(ctx, J, np.zeros(1024), L.PREC_AUTO), L.Model.sparse(ctx, sp.csc_matrix(J), np.zeros(1024))):
        e = L.Ensemble(model, 64)
        e.set_spins(S0)
        out = e.ssf_run(L.RULE_METROPOLIS, 8 * 1024, seed=9, T=T, steps_per_T=1024, trace_every=1024)
        res.append((e.get_spins(), out["flips"], out["E"]))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])
    assert _close(res[0][2], res[1][2])


def test_reference_style_sparse_system(pkg, ctx):
    """SpinSystem built from a scipy sparse matrix (the reference's tests use sparse(...)) stays sparse on the GPU."""
    import scipy.sparse as sp
    ss = pkg.SpinSystems.SpinSystem([-1, +1], sp.csc_matrix(np.array([[0, 1], [1, 0]])), [0, 0])
    assert pkg.SpinSystems.calcEnergy(ss) == 1.0
    assert ss._model.kind == "sparse"
    ua = pkg.SingleSpinFlip.GlauberDynamics(ss, 0.0)
    pkg.SingleSpinFlip.update_(ua, 0, 0.0)
    assert ss.spinConfiguration.tolist() == [1, 1] and pkg.SpinSystems.calcEnergy(ss) == -1.0


def test_dense_model_above_1024_sites(ctx, orc, synth):
    """Dense J with N > 1024 runs through the neighbour-list kernel (no ISB_ERR_UNSUPPORTED)."""
    L = _lib()
    n, R, nsteps = 1500, 6, 1500 * 2
    J, h = synth.sk_J(n, 3), synth.gaussian(4, n) * 0.1
    S0 = synth.spins(5, R, n)
    fl = synth.logistic(6, (R, nsteps))
    T = np.array([1.5, 0.5])
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    out = e.ssf_run(1, nsteps, fluct=fl, fluct_per_replica=True, T=T, steps_per_T=n, trace_every=n)
    S = e.get_spins()
    for r in range(R):
        s, flips, E, M = orc.ssf_run(1, J, h, S0[r], nsteps, fluct=fl[r], T=T, steps_per_T=n, trace_every=n)
        assert np.array_equal(s, S[r]) and flips == out["flips"][r] and _close(out["E"][:, r], E)
    assert _close(e.energy(), np.array([orc.energy(J, h, S[r]) for r in range(R)]))


@pytest.mark.parametrize("path,rule", [("dense", 2), ("dense", 1), ("sparse", 2), ("sparse", 1), ("f32", 1)])
def test_energy_distribution_matches_exact_result(ctx, synth, path, rule):
    """Independent RNG (in-kernel Philox): the mean energy of the 16 x 16 torus at T = 2.269 sampled by 4096
    chains of sequential sweeps agrees with Kaufman's exact finite-size value (tolerance: 5 standard errors
    estimated from the replica scatter + 0.1 % for the residual equilibration bias).  Path f32: the dense Float32 kernels
    (float couplings and fields), which must sample the Boltzmann distribution of the float couplings (here exact)."""
    import scipy.sparse as sp
    from exact_ising import mean_energy
    L_, T, R = 16, 2.269, 4096
    N = L_ * L_
    L = _lib()
    J = synth.lattice_J(L_)
    if path == "sparse":
        model = L.Model.sparse(ctx, sp.csc_matrix(J), np.zeros(N))
    else:
        model = L.Model.dense(ctx, J, np.zeros(N), L.PREC_F32 if path == "f32" else L.PREC_AUTO)
    e = L.Ensemble(model, R)
    e.set_spins(synth.spins(3, R, N))
    e.ssf_run(rule, 600 * N, seed=11, T=np.array([T]), steps_per_T=600 * N)            # equilibrate
    out = e.ssf_run(rule, 200 * N, seed=11, step_offset=600 * N, T=np.array([T]), steps_per_T=200 * N, trace_every=10 * N)
    Em = out["E"].mean(0)                       # time average per replica
    exact = mean_energy(L_, T)
    err = Em.std() / np.sqrt(R)
    assert abs(Em.mean() - exact) < 5 * err + 1e-3 * abs(exact), (Em.mean(), exact, err)


def test_per_replica_temperatures_bit_exact(ctx, orc, synth):
    """isb_ens_set_temperature_scale: replica r runs at Tsched * scale[r]; each replica equals the oracle run at
    that temperature (dense, sparse and Float64 bipartite kernels)."""
    import scipy.sparse as sp
    L = _lib()
    N, R, nsteps = 64, 9, 64 * 5
    J, h = synth.sk_J(N, 21), synth.gaussian(22, N) * 0.1
    S0 = synth.spins(23, R, N)
    fl = synth.logistic(24, (R, nsteps))
    T = synth.geometric_schedule(1.5, 0.5, 5)
    scale = np.linspace(0.4, 2.0, R)
    for model in (L.Model.dense(ctx, J, h, L.PREC_F64), L.Model.sparse(ctx, sp.csc_matrix(J), h)):
        e = L.Ensemble(model, R)
        e.set_spins(S0)
        e.set_temperature_scale(scale)
        out = e.ssf_run(1, nsteps, fluct=fl, fluct_per_replica=True, T=T, steps_per_T=N)
        S = e.get_spins()
        for r in range(R):
            s, flips, *_ = orc.ssf_run(1, J, h, S0[r], nsteps, fluct=fl[r], T=T * scale[r], steps_per_T=N)
            assert np.array_equal(s, S[r]) and flips == out["flips"][r]
        e.set_temperature_scale(None)   # cleared: back to the shared schedule
        e.set_spins(S0)
        e.ssf_run(1, nsteps, fluct=fl, fluct_per_replica=True, T=T, steps_per_T=N)
        s, *_ = orc.ssf_run(1, J, h, S0[0], nsteps, fluct=fl[0], T=T, steps_per_T=N)
        assert np.array_equal(s, e.get_spins()[0])
    nv, nh = 40, 24
    W, hv, bh = synth.bipartite_W(nv, nh, 25, 0.4)
    Sv, Sh = synth.spins(26, R, nv), synth.spins(27, R, nh)
    Fv, Fh = synth.logistic(28, (R, 3, nv), 1), synth.logistic(28, (R, 3, nh), 2)
    e = L.Ensemble(L.Model.bipartite(ctx, W, hv, bh, L.PREC_F64), R)
    e.set_spins(Sv)
    e.set_hidden(Sh)
    e.set_temperature_scale(scale)
    e.bip_run(0, 3, Fv=Fv, Fh=Fh, fluct_per_replica=True, T=np.array([1.0, 0.8, 0.6]))
    for r in range(R):
        s, t, _ = orc.bip_run(0, W, hv, bh, Sv[r], Sh[r], 3, Fv[r], Fh[r], np.array([1.0, 0.8, 0.6]) * scale[r])
        assert np.array_equal(s, e.get_spins()[r]) and np.array_equal(t, e.get_hidden()[r])
    # tensor-core path with integer couplings: per-replica temperatures, exact against the Float64 path
    Wi = np.round(W * 6.0)
    res = []
    for prec in (L.PREC_F64, L.PREC_BF16X1):
        e = L.Ensemble(L.Model.bipartite(ctx, Wi, np.round(hv * 6), np.round(bh * 6), prec), R)
        e.set_spins(Sv)
        e.set_hidden(Sh)
        e.set_temperature_scale(scale)
        e.bip_run(0, 3, Fv=Fv, Fh=Fh, fluct_per_replica=True, T=np.array([2.0, 1.5, 1.0]))
        res.append((e.get_spins(), e.get_hidden()))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])


def test_parallel_tempering_samples_each_temperature(pkg, ctx, synth):
    """Replica exchange on the 8 x 8 torus: the mean energy found at every temperature level agrees with Kaufman's
    exact value, and temperatures really travel between replicas."""
    import scipy.sparse as sp
    from exact_ising import mean_energy
    Lside, levels, ladders = 8, np.array([1.9, 2.2, 2.5, 2.9, 3.5]), 200
    N, R = Lside * Lside, ladders * 5
    ss = pkg.SpinSystems.SpinSystem(synth.spins(31, R, N), sp.csc_matrix(synth.lattice_J(Lside)), np.zeros(N))
    ua = pkg.SingleSpinFlip.MetropolisMethod(ss, 1.0)
    pt = pkg.tempering.ParallelTempering(ua, levels, seed=5)
    pt.run(150, sweeps=2)                       # equilibrate
    E = pt.run(150, sweeps=2)                   # [rounds][levels][ladders]
    assert (pt.accepted > 0).all() and (pt.accepted < pt.proposed).all()
    for lvl, T in enumerate(levels):
        per_ladder = E[:, lvl, :].mean(0)
        err = per_ladder.std() / np.sqrt(ladders)
        exact = mean_energy(Lside, T)
        assert abs(per_ladder.mean() - exact) < 5 * err + 2e-3 * abs(exact), (T, per_ladder.mean(), exact, err)


def test_configuration_histogram(pkg, ctx, synth):
    """demo.jl:159-168: the frequency of each spin configuration under Glauber dynamics at T = N/4 on the 3 x 3
    periodic antiferromagnet.  The device histogram equals the histogram of the recorded snapshots bit for bit
    (both counting paths), and the frequencies are the Boltzmann distribution."""
    L = _lib()
    tp = pkg.tempering
    assert tp.configurationIndex(np.array([[1, 1, -1], [-1, 1, 1]])).tolist() == [1, 4]
    for n, R in ((9, 64), (14, 48)):          # shared-memory bins / global atomics
        J = synth.lattice_J(3, -1.0) if n == 9 else synth.sk_J(n, 41)
        e = L.Ensemble(L.Model.dense(ctx, J, np.zeros(n), L.PREC_F64), R)
        S0 = synth.spins(42, R, n)
        e.set_spins(S0)
        out = e.ssf_run(1, 600, order=L.ORDER_RANDOM, seed=7, T=np.array([2.0]), steps_per_T=600, trace_every=3, want_S=True)
        want = np.bincount(tp.configurationIndex(out["S"]).ravel(), minlength=1 << n)
        e.set_spins(S0)
        hist = np.zeros(1 << n, dtype=np.int64)
        e.ssf_run(1, 600, order=L.ORDER_RANDOM, seed=7, T=np.array([2.0]), steps_per_T=600, trace_every=3, hist=hist)
        assert np.array_equal(hist, want) and hist.sum() == 200 * R
    n, R, T = 9, 512, 9 / 4
    J = synth.lattice_J(3, -1.0)
    ss = pkg.SpinSystems.SpinSystem(synth.spins(43, R, n), J, np.zeros(n))
    hist = tp.configurationHistogram(pkg.SingleSpinFlip.GlauberDynamics(ss, T), 9 * 400, stride=9, burn_in=9 * 50, seed=3)
    assert hist.sum() == 400 * R
    states = 1 - 2 * ((np.arange(512)[:, None] >> np.arange(8, -1, -1)) & 1)       # index -> spins, site 0 = MSB
    E = -0.5 * np.einsum("ki,ij,kj->k", states, J, states)
    p = np.exp(-E / T)
    p /= p.sum()
    tv = 0.5 * np.abs(hist / hist.sum() - p).sum()
    assert tv < 0.05, tv
    assert 0.5 * np.abs(1 / 512 - p).sum() > 0.2       # the target is far from uniform, so the bound above is a real check


def test_fields_in_global_memory_variant(ctx, orc, synth, monkeypatch):
    """Models whose fields do not fit the shared memory (N above ~25 000 sites) keep them in global memory; the variant is
    forced here on a small model and must follow the oracle bit for bit, then a 40 000-site random graph runs through it
    (traced energies against isb_ens_energy)."""
    L = _lib()
    monkeypatch.setenv("ISB_SPARSE_GLOBAL", "1")
    n, R, nsteps = 600, 9, 600 * 3 + 5
    A = _random_sparse(synth, n, 6, 300, False)
    J, h = A.toarray(), synth.gaussian(5, n) * 0.3
    S0 = synth.spins(6, R, n)
    fl = synth.logistic(8, (R, nsteps))
    T = synth.geometric_schedule(2.0, 0.2, 4)
    spT = (nsteps + 3) // 4
    for order in ("seq", "list"):
        nodes = synth.nodes(7, n, nsteps) if order == "list" else None
        e = L.Ensemble(L.Model.sparse(ctx, A, h), R)
        e.set_spins(S0)
        out = e.ssf_run(1, nsteps, nodes=nodes, start=17 if order == "seq" else 0, fluct=fl, fluct_per_replica=True, T=T,
                        steps_per_T=spT, trace_every=nsteps // 2)
        S = e.get_spins()
        for r in range(R):
            s, flips, E, M = orc.ssf_run(1, J, h, S0[r], nsteps, nodes=nodes, start=17 if order == "seq" else 0, fluct=fl[r], T=T,
                                         steps_per_T=spT, trace_every=nsteps // 2)
            assert np.array_equal(s, S[r]) and flips == out["flips"][r] and _close(out["E"][:, r], E)
    monkeypatch.delenv("ISB_SPARSE_GLOBAL")
    n, R = 40000, 3                                        # 9 N bytes = 360 kB per chain: beyond the shared memory
    A = _random_sparse(synth, n, 4, 301, True)
    e = L.Ensemble(L.Model.sparse(ctx, A, np.zeros(n)), R)
    e.set_spins(synth.spins(9, R, n))
    E0 = e.energy()
    out = e.ssf_run(2, 2 * n, seed=3, T=np.array([0.5]), steps_per_T=2 * n, trace_every=2 * n)
    assert _close(out["E"][-1], e.energy()) and np.all(e.energy() < E0)
