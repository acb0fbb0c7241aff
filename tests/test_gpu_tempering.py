"""GPU tests of device-resident parallel tempering (isb_ssf_run_pt, tempering.DeviceParallelTempering).

The core check is a replay: every round of isb_ssf_run_pt is by definition one isb_ssf_run of the same steps at the
replicas' current temperature factors, followed by one exchange whose rule (pairs, energies, Philox word, acceptance) is
reproduced in numpy here.  Spins, level assignments, traced E / M, overlaps, acceptance counts and flip totals must be
identical."""
import numpy as np
import pytest

from oracle.oracle_np import philox4x32_10

pytestmark = pytest.mark.gpu

DOM_PT_SWAP = 5


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


def _permuted_levels(seed, G, L):
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.permutation(L) for _ in range(G)]).astype(np.int32)


def exchange(lvl, Er, levels, K, seed, near):
    """One exchange of the documented rule on the host; lvl [R] is updated in place.  Returns accepted per pair.
    Decisions with |u - exp(d)| < 1e-12 (where libm and the device exp could disagree) are appended to `near`."""
    L = len(levels)
    G = len(lvl) // L
    rep = np.arange(G)[:, None] * L + np.argsort(lvl.reshape(G, L), axis=1)     # rep[g, l] = replica holding level l
    inv = 1.0 / levels
    acc = np.zeros(max(L - 1, 0), dtype=np.int64)
    for lo in range(K & 1, L - 1, 2):
        a, b = rep[:, lo], rep[:, lo + 1]
        d = (inv[lo] - inv[lo + 1]) * (Er[a] - Er[b])
        w = philox4x32_10(np.uint32(K & 0xFFFFFFFF), np.uint32(K >> 32), np.arange(G, dtype=np.uint32),
                          np.uint32((DOM_PT_SWAP << 28) | lo), seed & 0xFFFFFFFF, seed >> 32)[0]
        u = (w.astype(np.float64) + 0.5) * (1.0 / 4294967296.0)
        ex = np.exp(np.minimum(d, 0.0))
        near.extend((K, lo, int(g)) for g in np.nonzero((d < 0) & (np.abs(u - ex) < 1e-12))[0])
        ok = (d >= 0) | (u < ex)
        acc[lo] = int(ok.sum())
        lvl[a[ok]], lvl[b[ok]] = lo + 1, lo
    return acc


def replay(ens, rule, levels, rounds, spr, *, order, start, seed, step_offset, round_offset, level_of, want_Q):
    """isb_ssf_run_pt rebuilt from isb_ssf_run calls and the host exchange."""
    L = _lib()
    R, n = ens.R, ens.nv
    NL = len(levels)
    G = R // NL
    lvl = np.array(level_of, dtype=np.int32)
    E, M = np.zeros((rounds, NL, G)), np.zeros((rounds, NL, G))
    Q = np.zeros((rounds, NL, G // 2))
    acc, flips, near = np.zeros(max(NL - 1, 0), dtype=np.int64), np.zeros(R, dtype=np.int64), []
    for k in range(rounds):
        ens.set_temperature_scale(levels[lvl])
        out = ens.ssf_run(rule, spr, order=order, start=(start + k * spr) % n, seed=seed, step_offset=step_offset + k * spr,
                          T=np.array([1.0]), steps_per_T=spr, trace_every=spr)
        Er, Mr = out["E"][0], out["M"][0]
        flips += out["flips"]
        rep = np.arange(G)[:, None] * NL + np.argsort(lvl.reshape(G, NL), axis=1)
        E[k], M[k] = Er[rep].T, Mr[rep].T
        if want_Q:
            S = ens.get_spins().astype(np.int64)
            for p in range(G // 2):
                Q[k, :, p] = (S[rep[2 * p]] * S[rep[2 * p + 1]]).sum(1) / n
        acc += exchange(lvl, Er, levels, round_offset + k, seed, near)
    return {"level_of": lvl, "E": E, "M": M, "Q": Q if want_Q else None, "accepted": acc, "flips": flips}, near


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


# (model, rule, order, levels, ladders, rounds, steps per round as a multiple of N or an absolute count, start)
CASES = [
    ("sk64_f64", 1, "seq", 6, 4, 9, 40, 5),             # rounds shorter than N
    ("sk64_f64", 2, "seq", 5, 2, 7, 64, 0),             # equal to N, odd number of levels
    ("sk64_f64", 1, "seq", 6, 4, 5, 150, 63),           # longer than N
    ("sk64_f32", 2, "seq", 4, 6, 8, 64, 3),
    ("sk64_f64", 1, "random", 6, 4, 6, 100, 0),
    ("sk64_f64", 2, "seq", 1, 8, 4, 50, 7),             # one level: rounds without swaps
    ("dense1500", 1, "seq", 4, 2, 5, 1000, 17),         # N > 1024: the neighbour-list path
    ("sparse300", 2, "seq", 6, 4, 6, 450, 11),
    ("sparse300", 1, "seq", 6, 4, 6, 300, 0),
    ("lattice32", 2, "seq", 6, 4, 6, 1024, 0),
    ("lattice32", 2, "checkerboard", 6, 4, 5, 1500, 100),
    ("lattice32", 1, "checkerboard", 4, 2, 6, 700, 0),
]


@pytest.mark.parametrize("kind,rule,order,NL,G,rounds,spr,start", CASES)
def test_replay_parity(ctx, synth, kind, rule, order, NL, G, rounds, spr, start):
    L = _lib()
    o = {"seq": L.ORDER_SEQUENTIAL, "random": L.ORDER_RANDOM, "checkerboard": L.ORDER_CHECKERBOARD}[order]
    model, n = _model(ctx, synth, kind)
    R = NL * G
    # adjacent levels 1.5 / sqrt(N) apart (relative): close enough for swaps to be accepted at every model size
    T0 = {"sparse300": 3.0, "lattice32": 2.1}.get(kind, 0.8)
    levels = T0 * (1.0 + 1.5 / np.sqrt(n)) ** np.arange(NL)
    S0 = synth.spins(21, R, n)
    lvl0 = _permuted_levels(22, G, NL)
    seed, off, roff = 0x1234ABCD5678, 977, 5
    a, b = L.Ensemble(model, R), L.Ensemble(model, R)
    a.set_spins(S0)
    b.set_spins(S0)
    got = a.ssf_run_pt(rule, levels, rounds, spr, order=o, start=start, seed=seed, step_offset=off, round_offset=roff,
                       level_of=lvl0, want_E=True, want_M=True, want_Q=G % 2 == 0)
    want, near = replay(b, rule, levels, rounds, spr, order=o, start=start, seed=seed, step_offset=off, round_offset=roff,
                        level_of=lvl0, want_Q=G % 2 == 0)
    if near:
        pytest.skip(f"decisions within 1e-12 of exp(d) (libm vs device exp): {near}")
    assert np.array_equal(a.get_spins(), b.get_spins())
    assert np.array_equal(got["level_of"], want["level_of"])
    assert np.array_equal(got["E"], want["E"]) and np.array_equal(got["M"], want["M"])
    if G % 2 == 0:
        assert np.array_equal(got["Q"], want["Q"])
    assert np.array_equal(got["accepted"], want["accepted"])
    assert np.array_equal(got["flips"], want["flips"])
    st = a.last_stats()
    assert st["flips"] == int(want["flips"].sum()) and st["launches"] >= 2 * rounds and st["kernel_ms"] > 0
    if NL > 1:
        assert want["accepted"].sum() > 0          # the case exercises real swaps
    # the ensemble keeps the final ladder: a plain run continues both identically
    b.set_temperature_scale(levels[want["level_of"]])
    ra = a.ssf_run(rule, 2 * n, seed=3, T=np.array([1.0]), steps_per_T=2 * n, trace_every=n)
    rb = b.ssf_run(rule, 2 * n, seed=3, T=np.array([1.0]), steps_per_T=2 * n, trace_every=n)
    assert np.array_equal(a.get_spins(), b.get_spins()) and np.array_equal(ra["E"], rb["E"])


def test_oracle_anchor(ctx, orc, synth):
    """Integer couplings (+-1 SK, N = 24, 3 ladders x 4 levels): every replica of every round equals the CPU oracle run
    at that replica's temperature with the library's Philox fluctuations; the swaps follow the oracle's energies."""
    L = _lib()
    n, NL, G, rounds, spr, start, seed = 24, 4, 3, 8, 30, 5, 99
    J = np.sign(synth.sk_J(n, 31))
    h = np.zeros(n)
    levels = np.array([0.7, 1.1, 1.7, 2.6])
    R = NL * G
    S0 = synth.spins(32, R, n)
    lvl0 = np.tile(np.arange(NL, dtype=np.int32), G)
    for rule in (L.RULE_GLAUBER, L.RULE_METROPOLIS):
        e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
        e.set_spins(S0)
        got = e.ssf_run_pt(rule, levels, rounds, spr, start=start, seed=seed, level_of=lvl0, want_M=True)
        S, lvl, near = S0.copy(), lvl0.copy(), []
        for k in range(rounds):
            Er, Mr = np.zeros(R), np.zeros(R)
            for r in range(R):
                fl = ctx.philox_fluct(rule, seed, k * spr, r, 1, spr)[0]
                S[r], _, Et, Mt = orc.ssf_run(rule, J, h, S[r], spr, start=(start + k * spr) % n, fluct=fl,
                                              T=np.array([levels[lvl[r]]]), steps_per_T=spr, trace_every=spr)
                Er[r], Mr[r] = Et[0], Mt[0]
            rep = np.arange(G)[:, None] * NL + np.argsort(lvl.reshape(G, NL), axis=1)
            assert np.array_equal(got["E"][k], Er[rep].T) and np.array_equal(got["M"][k], Mr[rep].T), k
            exchange(lvl, Er, levels, k, seed, near)
        assert not near
        assert np.array_equal(e.get_spins(), S) and np.array_equal(got["level_of"], lvl)


def test_two_calls_equal_one(ctx, synth):
    """K + K rounds (start, step_offset and round_offset continued) equal 2K rounds bit for bit."""
    L = _lib()
    model = L.Model.dense(ctx, synth.sk_J(64, 41), None, L.PREC_F64)
    NL, G, K, spr, n = 6, 4, 7, 48, 64
    levels = np.geomspace(0.5, 2.0, NL)
    S0 = synth.spins(42, NL * G, n)
    a, b = L.Ensemble(model, NL * G), L.Ensemble(model, NL * G)
    a.set_spins(S0)
    b.set_spins(S0)
    lvl0 = _permuted_levels(43, G, NL)
    one = a.ssf_run_pt(1, levels, 2 * K, spr, start=9, seed=7, step_offset=100, round_offset=3, level_of=lvl0,
                       want_M=True, want_Q=True)
    p1 = b.ssf_run_pt(1, levels, K, spr, start=9, seed=7, step_offset=100, round_offset=3, level_of=lvl0,
                      want_M=True, want_Q=True)
    p2 = b.ssf_run_pt(1, levels, K, spr, start=(9 + K * spr) % n, seed=7, step_offset=100 + K * spr, round_offset=3 + K,
                      level_of=p1["level_of"], want_M=True, want_Q=True)
    assert np.array_equal(a.get_spins(), b.get_spins())
    assert np.array_equal(one["level_of"], p2["level_of"])
    for key in ("E", "M", "Q"):
        assert np.array_equal(one[key], np.concatenate([p1[key], p2[key]])), key
    assert np.array_equal(one["accepted"], p1["accepted"] + p2["accepted"])
    assert np.array_equal(one["flips"], p1["flips"] + p2["flips"])
    # a plain run after the call continues at the stored factors levels[level_of]
    c = L.Ensemble(model, NL * G)
    c.set_spins(a.get_spins())
    c.set_temperature_scale(levels[one["level_of"]])
    ra = a.ssf_run(1, 3 * n, seed=8, T=np.array([1.0]), steps_per_T=3 * n, trace_every=n)
    rc = c.ssf_run(1, 3 * n, seed=8, T=np.array([1.0]), steps_per_T=3 * n, trace_every=n)
    assert np.array_equal(a.get_spins(), c.get_spins()) and np.array_equal(ra["E"], rc["E"])


def test_device_class_matches_host_bookkeeping(pkg, ctx, synth):
    """DeviceParallelTempering: run() continues across calls like one call, keeps level / accepted / proposed, marks the
    host spins stale and leaves the ladder's factors for a later plain run."""
    n, NL, G = 64, 5, 4
    J = synth.sk_J(n, 51)
    levels = np.geomspace(0.5, 2.0, NL)
    pts = []
    for split in ((10,), (3, 7)):
        ss = pkg.SpinSystems.SpinSystem(synth.spins(52, NL * G, n), J, np.zeros(n))
        pt = pkg.tempering.DeviceParallelTempering(pkg.SingleSpinFlip.GlauberDynamics(ss, 1.0), levels, seed=4)
        parts = [pt.run(r, sweeps=2, overlaps=True) for r in split]
        pts.append((pt, ss, np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])))
    (p1, s1, E1, Q1), (p2, s2, E2, Q2) = pts
    assert E1.shape == (10, NL, G) and Q1.shape == (10, NL, G // 2)
    assert np.array_equal(E1, E2) and np.array_equal(Q1, Q2)
    assert np.array_equal(s1.spinConfiguration, s2.spinConfiguration)
    assert np.array_equal(p1.level, p2.level) and np.array_equal(p1.accepted, p2.accepted)
    assert np.array_equal(p1.proposed, p2.proposed)
    assert p1.proposed.tolist() == [G * 5] * (NL - 1)          # 10 rounds: 5 of each parity
    assert np.array_equal(np.sort(p1.level, axis=1), np.tile(np.arange(NL), (G, 1)))
    assert np.array_equal(p1.ua.temperatureScale, levels[p1.level].reshape(-1))
    # the energies it reports are those of the spins it leaves (last round, level l of ladder g)
    Ecur = pkg.SpinSystems.calcEnergy(p1.ua)
    assert np.all(np.abs(np.sort(np.asarray(Ecur).reshape(G, NL), axis=1) -
                         np.sort(E1[-1].T, axis=1)) <= 1e-9 * np.maximum(1.0, np.abs(E1[-1].T)))


def test_lattice_mean_energy_per_level(pkg, ctx, synth):
    """32 x 32 torus, lattice kernel, Metropolis, six levels around T_c, 64 ladders: the mean energy at every level
    agrees with Kaufman's exact value; every level pair swaps, and not always."""
    import scipy.sparse as sp
    from exact_ising import mean_energy
    Lside, levels, ladders = 32, np.array([2.0, 2.12, 2.24, 2.36, 2.5, 2.65]), 64
    N, R = Lside * Lside, ladders * len(levels)
    ss = pkg.SpinSystems.SpinSystem(np.ones((R, N), dtype=np.int8), sp.csc_matrix(synth.lattice_J(Lside)), np.zeros(N))
    pt = pkg.tempering.DeviceParallelTempering(pkg.SingleSpinFlip.MetropolisMethod(ss, 1.0), levels, seed=5)
    pt.run(3000)                                # equilibrate
    E = pt.run(3000)                            # [rounds][levels][ladders]
    assert (pt.accepted > 0).all() and (pt.accepted < pt.proposed).all()
    for lvl, T in enumerate(levels):
        per_ladder = E[:, lvl, :].mean(0)
        err = per_ladder.std() / np.sqrt(ladders)
        exact = mean_energy(Lside, T)
        assert abs(per_ladder.mean() - exact) < 5 * err + 2e-3 * abs(exact), (T, per_ladder.mean(), exact, err)


def test_dense_mean_energy_matches_enumeration(pkg, ctx, synth):
    """Dense N = 12 model with fields: the mean energy at every level equals the Boltzmann average by enumeration."""
    n, levels, ladders = 12, np.array([0.6, 0.9, 1.35, 2.0]), 64
    J, h = synth.sk_J(n, 61) * 2.0, synth.gaussian(62, n) * 0.3
    ss = pkg.SpinSystems.SpinSystem(synth.spins(63, ladders * len(levels), n), J, h)
    pt = pkg.tempering.DeviceParallelTempering(pkg.SingleSpinFlip.GlauberDynamics(ss, 1.0), levels, seed=6)
    pt.run(300)
    E = pt.run(4000)
    assert (pt.accepted > 0).all() and (pt.accepted < pt.proposed).all()
    states = 1 - 2 * ((np.arange(1 << n)[:, None] >> np.arange(n)) & 1)
    Es = -0.5 * np.einsum("ki,ij,kj->k", states, J, states) - states @ h
    for lvl, T in enumerate(levels):
        w = np.exp(-(Es - Es.min()) / T)
        exact = float((Es * w).sum() / w.sum())
        per_ladder = E[:, lvl, :].mean(0)
        err = per_ladder.std() / np.sqrt(ladders)
        assert abs(per_ladder.mean() - exact) < 5 * err + 2e-3 * abs(exact), (T, per_ladder.mean(), exact, err)


def test_errors_leave_the_ensemble_unchanged(ctx, synth):
    L = _lib()
    n, NL, G = 32, 4, 3
    model = L.Model.dense(ctx, synth.sk_J(n, 71), None, L.PREC_F64)
    e = L.Ensemble(model, NL * G)
    S0 = synth.spins(72, NL * G, n)
    e.set_spins(S0)
    e.set_temperature_scale(np.linspace(0.5, 1.5, NL * G))
    ref = e.clone()
    levels = np.array([0.5, 0.8, 1.2, 2.0])
    lvl = np.tile(np.arange(NL, dtype=np.int32), G)

    def expect(code, *args, ens=e, **kw):
        kw.setdefault("level_of", lvl)
        before = np.array(kw["level_of"], copy=True)
        with pytest.raises(L.IsbError) as ei:
            ens.ssf_run_pt(*args, **kw)
        assert ei.value.code == code and ei.value.message, (code, ei.value)
        assert np.array_equal(kw["level_of"], before)

    W, hv, hb = synth.bipartite_W(8, 4, 73)
    bip = L.Ensemble(L.Model.bipartite(ctx, W, hv, hb), NL * G)
    expect(L.ERR_STATE, 1, levels, 2, n, ens=bip)
    expect(L.ERR_ARG, L.RULE_HOPFIELD, levels, 2, n)
    expect(L.ERR_ARG, 1, levels, 2, n, order=L.ORDER_LIST)
    expect(L.ERR_SIZE, 1, np.array([0.5, 0.8, 1.2, 2.0, 3.0]), 2, n, level_of=np.zeros(NL * G, dtype=np.int32))
    expect(L.ERR_ARG, 1, np.zeros(0), 2, n, level_of=np.zeros(NL * G, dtype=np.int32))
    expect(L.ERR_UNSUPPORTED, 1, np.ones(1025), 2, n, level_of=np.zeros(NL * G, dtype=np.int32))
    expect(L.ERR_NONFINITE, 1, np.array([0.5, np.nan, 1.2, 2.0]), 2, n)
    expect(L.ERR_NONFINITE, 1, np.array([0.5, 0.8, np.inf, 2.0]), 2, n)
    expect(L.ERR_ARG, 1, np.array([0.5, 0.0, 1.2, 2.0]), 2, n)
    expect(L.ERR_ARG, 1, np.array([0.5, -0.8, 1.2, 2.0]), 2, n)
    bad = lvl.copy()
    bad[5] = bad[4]
    expect(L.ERR_ARG, 1, levels, 2, n, level_of=bad)
    bad = lvl.copy()
    bad[0] = NL
    expect(L.ERR_ARG, 1, levels, 2, n, level_of=bad)
    expect(L.ERR_SIZE, 1, levels, 2, n, want_Q=True)              # three ladders
    expect(L.ERR_ARG, 1, levels, 2, 0)
    expect(L.ERR_ARG, 1, levels, 2, -5)
    # rounds = 0 is a no-op
    out = e.ssf_run_pt(1, levels, 0, n, level_of=lvl)
    assert np.array_equal(out["level_of"], lvl) and not out["flips"].any() and not out["accepted"].any()
    # nothing moved: spins and temperature factors are those of the clone taken before
    assert np.array_equal(e.get_spins(), S0)
    ra = e.ssf_run(1, 2 * n, seed=1, T=np.array([1.0]), steps_per_T=2 * n, trace_every=n)
    rb = ref.ssf_run(1, 2 * n, seed=1, T=np.array([1.0]), steps_per_T=2 * n, trace_every=n)
    assert np.array_equal(e.get_spins(), ref.get_spins()) and np.array_equal(ra["E"], rb["E"])
