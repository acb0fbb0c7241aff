"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI
(include/ising_b200.h via ctypes), against the CPU oracle on the same seeded inputs.

Bar: spin trajectories, flip counts and magnetisations BIT-EXACT; energies within 1e-9 relative (the
energy is a different summation order of the same Float64 quantities; north_star allows 1e-5)."""
import numpy as np
import pytest

from cases import BIP_GOLDEN, SSF_GOLDEN, golden_J, golden_W, nodes_of
from conftest import load_golden

pytestmark = pytest.mark.gpu
E_RTOL = 1e-9


def _close(a, b):
    scale = np.maximum(1.0, np.abs(b))
    return np.all(np.abs(a - b) <= E_RTOL * scale)


def _lib():
    from isingmodel_jl_b200 import _lib
    return _lib


# ---------------------------------------------------------------- Philox
def test_philox_raw_matches_oracle_and_kat(ctx, orc):
    kat_ctr = np.array([[0, 0, 0, 0], [0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]], dtype=np.uint32)
    got = ctx.philox_raw(kat_ctr[1:], np.array([0xa4093822, 0x299f31d0], dtype=np.uint32))
    assert got[0].tolist() == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    rng = np.random.default_rng(0)
    ctrs = rng.integers(0, 2 ** 32, (257, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2 ** 32, 2, dtype=np.uint64).astype(np.uint32)
    got = ctx.philox_raw(ctrs, key)
    want = np.array([orc.philox4x32_10(c, key) for c in ctrs])
    assert np.array_equal(got, want)


def test_philox_streams(ctx):
    from oracle import oracle_np
    L = _lib()
    seed, off = 0x1234567890ABCDEF, 5
    fl = ctx.philox_fluct(L.RULE_GLAUBER, seed, off, 3, 2, 64)
    steps = np.arange(64, dtype=np.uint64) + np.uint64(off)
    for i, r in enumerate((3, 4)):
        w = oracle_np.philox_word(seed, 1 << 28, r, steps)
        u = oracle_np.uniform_from_word(w)
        assert np.allclose(fl[i], np.log(u / (1 - u)), rtol=4e-6, atol=4e-6)  # variates evaluated in fp32 on the device
    fe = ctx.philox_fluct(L.RULE_METROPOLIS, seed, off, 0, 1, 64)
    u = oracle_np.uniform_from_word(oracle_np.philox_word(seed, 1 << 28, 0, steps))
    assert np.allclose(fe[0], -np.log(u), rtol=4e-6, atol=4e-6)
    nd = ctx.philox_nodes(1000, seed, off, 64)
    w = oracle_np.philox_word(seed, 2 << 28, 0, steps)
    assert np.array_equal(nd, ((w.astype(np.uint64) * np.uint64(1000)) >> np.uint64(32)).astype(np.int32))


# ---------------------------------------------------------------- golden files, R = 1 (the reference's one chain)
@pytest.mark.parametrize("name", SSF_GOLDEN)
def test_ssf_golden(ctx, synth, name):
    L = _lib()
    g = load_golden(name)
    J = golden_J(name, g, synth)
    m = L.Model.dense(ctx, J, g["h"], L.PREC_AUTO)
    e = L.Ensemble(m, 1)
    e.set_spins(g["s0"][None, :])
    out = e.ssf_run(int(g["rule"]), int(g["nsteps"]), nodes=nodes_of(g), fluct=g["fluct"], T=g["T"],
                    steps_per_T=int(g["steps_per_T"]), trace_every=int(g["trace_every"]))
    assert np.array_equal(e.get_spins()[0], g["s_final"])
    assert int(out["flips"][0]) == int(g["flips"])
    assert np.array_equal(out["M"][:, 0], g["M"])
    assert _close(out["E"][:, 0], g["E"])
    assert _close(e.energy()[0], g["E"][-1])


@pytest.mark.parametrize("name", BIP_GOLDEN)
def test_bip_golden(ctx, synth, name):
    L = _lib()
    g = load_golden(name)
    W = golden_W(name, g, synth)
    m = L.Model.bipartite(ctx, W, g["h"], g["b"], L.PREC_F64)
    e = L.Ensemble(m, 1)
    e.set_spins(g["s0"][None, :])
    e.set_hidden(g["t0"][None, :])
    E = e.bip_run(int(g["rule"]), int(g["nsteps"]), Fv=g["Fv"], Fh=g["Fh"], T=g["T"], trace_every=1)
    assert np.array_equal(e.get_spins()[0], g["s_final"])
    assert np.array_equal(e.get_hidden()[0], g["t_final"])
    assert _close(E[:, 0], g["E"])


# ---------------------------------------------------------------- replica-batched sweeps vs the oracle
SSF_CASES = [
    # (N, kind, rule, order, prec, R, nsteps, per_replica)
    (1, "sk", 1, "seq", "f64", 3, 7, True),
    (2, "sk", 2, "list", "f64", 3, 50, True),
    (31, "sk", 1, "seq", "f64", 5, 31 * 9 + 4, True),
    (32, "sk", 2, "list", "f64", 33, 700, True),
    (33, "sk", 1, "seq", "f64", 29, 33 * 7, False),
    (100, "sk", 2, "seq", "f64", 40, 100 * 6 + 17, True),
    (100, "sk", 0, "list", "f64", 4, 500, False),
    (256, "lattice", 2, "seq", "auto", 64, 256 * 8, True),
    (256, "lattice", 1, "list", "auto", 7, 3000, True),
    (500, "sk", 1, "seq", "f64", 200, 500 * 3, True),
    (1000, "sk", 2, "seq", "f64", 31, 1000 * 2 + 3, True),
    (1024, "sk", 1, "seq", "f64", 300, 1024 * 3, True),
    (1024, "lattice", 2, "seq", "auto", 300, 1024 * 4, True),
    (1024, "sk", 1, "list", "f64", 15, 4000, True),
    (1024, "sk", 0, "seq", "f64", 9, 2048, False),
]


def _ssf_inputs(synth, N, kind, rule, order, R, nsteps, per_replica, seed=1):
    if kind == "lattice":
        Lside = int(round(np.sqrt(N)))
        J = synth.lattice_J(Lside)
        h = np.zeros(N)
    else:
        J = synth.sk_J(N, seed + N)
        h = synth.gaussian(seed + 1, N) * 0.2
    S0 = synth.spins(seed + 2, R, N)
    nodes = synth.nodes(seed + 3, N, nsteps) if order == "list" else None
    shape = (R, nsteps) if per_replica else (nsteps,)
    fl = synth.logistic(seed + 4, shape) if rule == 1 else (synth.exponential(seed + 4, shape) if rule == 2 else None)
    nT = 7
    spT = (nsteps + nT - 1) // nT
    T = synth.geometric_schedule(2.5, 0.3, nT)
    return J, h, S0, nodes, fl, T, spT


@pytest.mark.parametrize("N,kind,rule,order,prec,R,nsteps,per_replica", SSF_CASES)
def test_ssf_batched_bit_exact(ctx, orc, synth, N, kind, rule, order, prec, R, nsteps, per_replica):
    L = _lib()
    J, h, S0, nodes, fl, T, spT = _ssf_inputs(synth, N, kind, rule, order, R, nsteps, per_replica)
    m = L.Model.dense(ctx, J, h, L.PREC_AUTO if prec == "auto" else L.PREC_F64)
    e = L.Ensemble(m, R)
    e.set_spins(S0)
    e.set_tie_eps(1e-12)
    tr = max(1, nsteps // 3)
    out = e.ssf_run(rule, nsteps, nodes=nodes, start=(N // 3) if order == "seq" else 0, fluct=fl,
                    fluct_per_replica=per_replica, T=T, steps_per_T=spT, trace_every=tr)
    S = e.get_spins()
    stats = e.last_stats()
    mism = 0
    for r in range(R):
        f = None if fl is None else (fl[r] if per_replica else fl)
        s, flips, E, M = orc.ssf_run(rule, J, h, S0[r], nsteps, nodes=nodes, start=(N // 3) if order == "seq" else 0,
                                     fluct=f, T=T, steps_per_T=spT, trace_every=tr)
        if not np.array_equal(s, S[r]):
            mism += 1
            continue
        assert flips == out["flips"][r]
        assert np.array_equal(M, out["M"][:, r])
        assert _close(out["E"][:, r], E)
    # Gaussian J: the incrementally maintained Float64 field differs from the oracle's fresh row sum by a few
    # ulp, so a decision can differ only where |2h - fT| is below ~1e-13; the kernel counts those (near-tie audit).
    assert mism == 0 or stats["near_ties"] > 0, f"{mism} replicas differ without any near tie"
    assert mism == 0
    assert stats["flips"] == int(out["flips"].sum())
    assert _close(e.energy(), np.array([orc.energy(J, h, S[r]) for r in range(R)]))
    assert np.array_equal(e.magnetization(), S.sum(1).astype(np.float64))


@pytest.mark.parametrize("thr", ["0.2", "0", "2"])
@pytest.mark.parametrize("rule,per_rep", [(1, True), (2, False)])
def test_ssf_segmented_run_equals_the_oracle(ctx, orc, synth, monkeypatch, thr, rule, per_rep):
    """Long sequential sweeps are run segment by segment, each launch with the streaming or the plain kernel according
    to the previous segment's acceptance (csrc/ssf.cu).  Forced here at a small size (3 sweeps per segment; threshold
    0.2 = the product's rule, 0 = always streaming, 2 = plain after the first segment): spins, flip counts and traces
    must equal the oracle's single run — noise, schedule entries, first site and trace slots are all indexed by the
    step of the whole run — and the single-launch run of the library."""
    L = _lib()
    N, R, sweeps, start = 96, 70, 41, 37
    nsteps = sweeps * N + 29                                  # the last segment is ragged
    J, h = synth.sk_J(N, 71), synth.gaussian(72, N) * 0.2
    S0 = synth.spins(73, R, N)
    gen = synth.logistic if rule == 1 else synth.exponential
    fl = gen(74, (R, nsteps) if per_rep else nsteps)
    T = synth.geometric_schedule(2.5, 0.05, sweeps + 1)       # hot to cold: both kernels get their turn at thr = 0.2
    tr = 2 * N
    runs = {}
    for seg in ("1", "0"):
        monkeypatch.setenv("ISB_SSF_SEGMENT", seg)
        monkeypatch.setenv("ISB_SSF_SEG_MIN", str(3 * N))
        monkeypatch.setenv("ISB_SSF_SEG_THR", thr)
        e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
        e.set_spins(S0)
        out = e.ssf_run(rule, nsteps, start=start, fluct=fl, fluct_per_replica=per_rep, T=T, steps_per_T=N, trace_every=tr,
                        want_S=True)
        runs[seg] = (e.get_spins(), out, e.last_stats()["launches"])
    S, out, launches = runs["1"]
    assert launches >= runs["0"][2] + 4                       # it really was segmented (cold segments double in length)
    assert np.array_equal(S, runs["0"][0]) and np.array_equal(out["flips"], runs["0"][1]["flips"])
    assert np.array_equal(out["E"], runs["0"][1]["E"]) and np.array_equal(out["S"], runs["0"][1]["S"])
    for r in (0, 1, R // 2, R - 1):
        s, flips, E, M = orc.ssf_run(rule, J, h, S0[r], nsteps, start=start, fluct=fl[r] if per_rep else fl, T=T,
                                     steps_per_T=N, trace_every=tr)
        assert np.array_equal(s, S[r]) and flips == out["flips"][r], f"replica {r}"
        assert np.array_equal(M, out["M"][:, r]) and _close(out["E"][:, r], E)


@pytest.mark.parametrize("fixed", ["1", "0"])
@pytest.mark.parametrize("rule,per_rep,start", [(1, True, 5), (2, False, 0), (0, False, 77)])
@pytest.mark.parametrize("thr,thr_cold", [(None, None), ("2", "2"), ("0.5", "0.25")])
def test_ssf_cold_kernel_in_segmented_runs(ctx, orc, synth, monkeypatch, thr, thr_cold, rule, per_rep, start, fixed):
    """The third kernel of a segmented run (csrc/ssf_cold.cu: fields in shared memory, 28 chains per SM), chosen when the
    previous segment accepted few flips and the run has no traces.  Untraced sequential runs take the fixed-point kernels
    (plain and cold, product thresholds 2.0 / 0.06); with ISB_SSF_FIXED=0 they take the Float64 ones (streaming, plain and
    cold, product thresholds 0.2 / 0.03).  Thresholds: the product's, "cold from the second segment on", and a mix that
    alternates the kernels.  The cached fields pass from kernel to kernel, so every replica must still equal the oracle's
    single run bit for bit."""
    L = _lib()
    N, R, sweeps = 128, 90, 37
    nsteps = sweeps * N + 51
    J, h = synth.sk_J(N, 81), synth.gaussian(82, N) * 0.2
    S0 = synth.spins(83, R, N)
    gen = synth.logistic if rule == 1 else synth.exponential
    fl = None if rule == 0 else gen(84, (R, nsteps) if per_rep else nsteps)
    T = synth.geometric_schedule(3.0, 0.03, sweeps + 1)
    monkeypatch.setenv("ISB_SSF_FIXED", fixed)
    monkeypatch.setenv("ISB_SSF_SEG_MIN", str(3 * N))
    if thr is not None:
        monkeypatch.setenv("ISB_SSF_SEG_THR", thr)
        monkeypatch.setenv("ISB_SSF_COLD_THR", thr_cold)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    out = e.ssf_run(rule, nsteps, start=start, fluct=fl, fluct_per_replica=per_rep, T=T, steps_per_T=N)
    S = e.get_spins()
    assert e.last_stats()["launches"] >= 5 or rule == 0      # (Hopfield runs have no schedule to cut at: one launch)
    assert _close(e.energy()[:4], np.array([orc.energy(J, h, S[r]) for r in range(4)]))
    for r in (0, 1, R // 2, R - 1):
        s, flips, _, _ = orc.ssf_run(rule, J, h, S0[r], nsteps, start=start,
                                     fluct=None if fl is None else (fl[r] if per_rep else fl), T=T, steps_per_T=N)
        assert np.array_equal(s, S[r]) and flips == out["flips"][r], f"replica {r}"
    # and the run continues from the cached fields the cold kernel left behind
    e.ssf_run(rule, 5 * N, start=(start + nsteps) % N, fluct=None if fl is None else fl[..., :5 * N], fluct_per_replica=per_rep,
              T=T[:5], steps_per_T=N)
    s, _, _, _ = orc.ssf_run(rule, J, h, S[0], 5 * N, start=(start + nsteps) % N,
                             fluct=None if fl is None else (fl[0, :5 * N] if per_rep else fl[:5 * N]), T=T[:5], steps_per_T=N)
    assert np.array_equal(s, e.get_spins()[0])


def test_ssf_continuation_and_field_cache(ctx, orc, synth):
    """Two runs back to back == one run (cached local fields stay valid); set_spins invalidates them."""
    L = _lib()
    N, R, n1, n2 = 200, 10, 500, 700
    J, h, S0, _, fl, _, _ = _ssf_inputs(synth, N, "sk", 1, "seq", R, n1 + n2, True)
    T = synth.geometric_schedule(2.0, 0.2, n1 + n2)  # one temperature per step
    m = L.Model.dense(ctx, J, h, L.PREC_F64)
    e = L.Ensemble(m, R)
    e.set_spins(S0)
    e.ssf_run(1, n1, fluct=fl[:, :n1].copy(), fluct_per_replica=True, T=T[:n1])
    S_mid = e.get_spins()
    e.ssf_run(1, n2, start=n1 % N, fluct=fl[:, n1:].copy(), fluct_per_replica=True, T=T[n1:])
    S_end = e.get_spins()
    for r in range(R):
        s, *_ = orc.ssf_run(1, J, h, S0[r], n1, fluct=fl[r, :n1], T=T)
        assert np.array_equal(s, S_mid[r])
        s, *_ = orc.ssf_run(1, J, h, S0[r], n1 + n2, fluct=fl[r], T=T)
        assert np.array_equal(s, S_end[r])
    e.set_spins(S0)  # must drop the cached fields
    e.ssf_run(1, 300, fluct=fl[:, :300].copy(), fluct_per_replica=True, T=T[:300])
    S = e.get_spins()
    for r in range(R):
        s, *_ = orc.ssf_run(1, J, h, S0[r], 300, fluct=fl[r, :300], T=T)
        assert np.array_equal(s, S[r])


def test_ssf_philox_mode_reproduces_with_dumped_fluctuations(ctx, orc, synth):
    """ISB_FLUCT_PHILOX: the trajectories equal the oracle's when it is fed the fluctuations the library
    dumps for the same (seed, offset) — the 'shared uniforms' parity of north_star."""
    L = _lib()
    N, R, nsteps, seed, off = 1024, 40, 3 * 1024, 99, 1000
    J = synth.sk_J(N, 2)
    h = np.zeros(N)
    S0 = synth.spins(3, R, N)
    T = np.array([1.5, 1.0, 0.5])
    for rule in (L.RULE_GLAUBER, L.RULE_METROPOLIS):
        m = L.Model.dense(ctx, J, h, L.PREC_F64)
        e = L.Ensemble(m, R)
        e.set_spins(S0)
        e.ssf_run(rule, nsteps, seed=seed, step_offset=off, T=T, steps_per_T=N)
        S = e.get_spins()
        fl = ctx.philox_fluct(rule, seed, off, 0, R, nsteps)
        for r in range(R):
            s, *_ = orc.ssf_run(rule, J, h, S0[r], nsteps, fluct=fl[r], T=T, steps_per_T=N)
            assert np.array_equal(s, S[r])
        # random site order drawn by the library
        e.set_spins(S0)
        e.ssf_run(rule, 2000, order=L.ORDER_RANDOM, seed=seed, step_offset=off, T=T, steps_per_T=N)
        nodes = ctx.philox_nodes(N, seed, off, 2000)
        S = e.get_spins()
        for r in range(0, R, 7):
            s, *_ = orc.ssf_run(rule, J, h, S0[r], 2000, nodes=nodes, fluct=fl[r, :2000], T=T, steps_per_T=N)
            assert np.array_equal(s, S[r])


def test_local_field_bit_exact(ctx, orc, synth):
    L = _lib()
    N, R = 300, 6
    J, h = synth.sk_J(N, 8), synth.gaussian(9, N)
    S = synth.spins(10, R, N)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S)
    F = e.local_field()
    for r in range(R):
        assert np.array_equal(F[r], orc.local_field(J, h, S[r]))  # same sequential Float64 row sums


# ---------------------------------------------------------------- bipartite, replica-batched
BIP_CASES = [(2, 3, 0, 5, 6, True), (17, 9, 1, 11, 5, True), (130, 70, 0, 37, 4, False), (784, 512, 0, 19, 3, True),
             (784, 512, 1, 9, 3, True), (257, 1030, 0, 8, 2, True)]


@pytest.mark.parametrize("nv,nh,rule,R,nsteps,per_replica", BIP_CASES)
def test_bip_batched_bit_exact(ctx, orc, synth, nv, nh, rule, R, nsteps, per_replica):
    L = _lib()
    W, h, b = synth.bipartite_W(nv, nh, 21, 0.3)
    S0, T0 = synth.spins(22, R, nv), synth.spins(23, R, nh)
    gen = synth.logistic if rule == 0 else synth.exponential
    shp = (R, nsteps) if per_replica else (nsteps,)
    Fv, Fh = gen(24, shp + (nv,), 1), gen(24, shp + (nh,), 2)
    T = synth.geometric_schedule(2.0, 0.2, nsteps)
    e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, L.PREC_F64), R)
    e.set_spins(S0)
    e.set_hidden(T0)
    E = e.bip_run(rule, nsteps, Fv=Fv, Fh=Fh, fluct_per_replica=per_replica, T=T, trace_every=1)
    S, Tm = e.get_spins(), e.get_hidden()
    for r in range(R):
        s, t, Eo = orc.bip_run(rule, W, h, b, S0[r], T0[r], nsteps, Fv[r] if per_replica else Fv,
                               Fh[r] if per_replica else Fh, T, want_E=True)
        assert np.array_equal(s, S[r]) and np.array_equal(t, Tm[r])
        assert _close(E[:, r], Eo)
    A, F = e.local_aux_bias(), e.local_field()
    for r in range(min(R, 3)):
        assert np.array_equal(A[r], orc.bip_aux_bias(W, b, S[r]))
        assert np.array_equal(F[r], orc.bip_local_field(W, h, Tm[r]))


def test_bip_philox_mode(ctx, orc, synth):
    L = _lib()
    nv, nh, R, nsteps, seed, off = 96, 40, 6, 5, 7, 3
    W, h, b = synth.bipartite_W(nv, nh, 31, 0.3)
    S0, T0 = synth.spins(32, R, nv), synth.spins(33, R, nh)
    T = np.full(nsteps, 0.8)
    for rule in (0, 1):
        e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, L.PREC_F64), R)
        e.set_spins(S0)
        e.set_hidden(T0)
        e.bip_run(rule, nsteps, seed=seed, step_offset=off, T=T)
        Fv = ctx.philox_bip_fluct(rule, seed, off, 0, nv, 0, R, nsteps)
        Fh = ctx.philox_bip_fluct(rule, seed, off, 1, nh, 0, R, nsteps)
        S, Tm = e.get_spins(), e.get_hidden()
        for r in range(R):
            s, t, _ = orc.bip_run(rule, W, h, b, S0[r], T0[r], nsteps, Fv[r], Fh[r], T)
            assert np.array_equal(s, S[r]) and np.array_equal(t, Tm[r])


# ---------------------------------------------------------------- errors cross the ABI as codes
def test_error_codes(ctx, synth):
    L = _lib()
    with pytest.raises(L.IsbError) as ei:
        L.Model.dense(ctx, np.array([[0.0, np.nan], [np.nan, 0.0]]), np.zeros(2))
    assert ei.value.code == L.ERR_NONFINITE
    m = L.Model.dense(ctx, synth.sk_J(8, 1), np.zeros(8))
    assert m.warn == 0
    e = L.Ensemble(m, 2)
    with pytest.raises(L.IsbError) as ei:
        e.set_spins(np.zeros((2, 8), dtype=np.int8))
    assert ei.value.code == L.ERR_ARG
    with pytest.raises(L.IsbError) as ei:
        e.ssf_run(1, 10, nodes=np.full(10, 8), fluct=np.zeros(10), T=np.ones(10))
    assert ei.value.code == L.ERR_ARG
    with pytest.raises(L.IsbError) as ei:
        e.ssf_run(1, 10, fluct=np.zeros(10), T=np.ones(3))
    assert ei.value.code == L.ERR_SIZE
    with pytest.raises(L.IsbError) as ei:
        e.bip_run(0, 1, T=np.ones(1))
    assert ei.value.code == L.ERR_STATE
    A = np.array([[1.0, 2.0, 3.0], [0.0, 5.0, 6.0], [0.0, 0.0, 9.0]])
    m2 = L.Model.dense(ctx, A, np.zeros(3))
    assert m2.warn == 3  # symmetrised from the upper triangle + diagonal dropped (SpinSystems.jl:31-38)
    e2 = L.Ensemble(m2, 1)
    e2.set_spins(np.array([[1, 1, 1]], dtype=np.int8))
    assert np.array_equal(e2.local_field()[0], [5.0, 8.0, 9.0])


# ---------------------------------------------------------------- tcgen05 path (bf16 split couplings, fp32 TMEM accumulation)
def _tc_step_check(L, ctx, orc, W, h, b, S0, T0, rule, prec, Fv, Fh, T, tol):
    """One block-Gibbs step from the same state on the tensor-core path and on the oracle.  The accumulators
    are fp32 (not the oracle's Float64), so a decision may differ only where the oracle's decision quantity
    |2(W's + b) - F T| is below `tol` (near tie); with exactly representable W (tol = 0) it must be bit-exact."""
    R, nv = S0.shape
    nh = T0.shape[1]
    e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, prec), R)
    e.set_spins(S0)
    e.set_hidden(T0)
    e.bip_run(rule, 1, Fv=Fv, Fh=Fh, fluct_per_replica=True, T=np.array([T]))
    S, Tm = e.get_spins(), e.get_hidden()
    bad = 0
    for r in range(R):
        aux = orc.bip_aux_bias(W, b, S0[r])
        ft = Fh[r, 0] * T * (T0[r] if rule == 1 else 1.0)
        xh = 2.0 * aux - ft
        t_or = np.where(xh < 0, -1, 1).astype(np.int8)
        dh = Tm[r] != t_or
        assert np.all(np.abs(xh[dh]) <= tol), (r, np.abs(xh[dh]).max())
        bad += int(dh.sum())
        # visible layer from the hidden layer the GPU actually produced
        fld = orc.bip_local_field(W, h, Tm[r])
        ftv = Fv[r, 0] * T * (S0[r] if rule == 1 else 1.0)
        xv = 2.0 * fld - ftv
        s_or = np.where(xv < 0, -1, 1).astype(np.int8)
        dv = S[r] != s_or
        assert np.all(np.abs(xv[dv]) <= tol), (r, np.abs(xv[dv]).max())
        bad += int(dv.sum())
    return bad, e


TC_CASES = [(64, 48, 0, 130, "x1int"), (784, 512, 0, 300, "x3"), (784, 512, 1, 200, "x3"), (200, 1000, 0, 257, "x3"),
            (784, 512, 0, 300, "x2"), (300, 260, 1, 140, "x2"),
            (96, 40, 1, 64, "x1int"), (1024, 1024, 0, 128, "x3")]


@pytest.mark.parametrize("nv,nh,rule,R,kind", TC_CASES)
def test_bip_tc_single_step(ctx, orc, synth, nv, nh, rule, R, kind):
    L = _lib()
    if kind == "x1int":  # small-integer couplings: exact in bf16, every partial sum exact in fp32
        W = np.round(synth.gaussian(71, nv * nh).reshape(nv, nh) * 2.0)
        h, b = np.round(synth.gaussian(72, nv)), np.round(synth.gaussian(73, nh))
        prec, tol = L.PREC_BF16X1, 0.0
    else:
        W, h, b = synth.bipartite_W(nv, nh, 74, 0.1)
        prec, tol = (L.PREC_BF16X3, 2e-4) if kind == "x3" else (L.PREC_BF16X2, 6e-4)
    S0, T0 = synth.spins(75, R, nv), synth.spins(76, R, nh)
    gen = synth.logistic if rule == 0 else synth.exponential
    Fv, Fh = gen(77, (R, 1, nv), 1), gen(77, (R, 1, nh), 2)
    bad, e = _tc_step_check(L, ctx, orc, W, h, b, S0, T0, rule, prec, Fv, Fh, 0.9, tol)
    assert bad <= max(2, int(1e-4 * R * (nv + nh)))
    if kind == "x1int":
        assert bad == 0
    # the canonical int8 state is what energy / field kernels see
    Eg = e.energy()
    S, Tm = e.get_spins(), e.get_hidden()
    Eo = np.array([orc.bip_energy(W, h, b, S[r], Tm[r]) for r in range(min(R, 8))])
    assert _close(Eg[:len(Eo)], Eo)


def test_bip_tc_exact_trajectory_integer_W(ctx, orc, synth):
    """Integer couplings: the tensor-core path is bit-exact, so whole trajectories match the oracle."""
    L = _lib()
    nv, nh, R, nsteps = 160, 96, 140, 6
    W = np.round(synth.gaussian(81, nv * nh).reshape(nv, nh) * 1.5)
    h, b = np.round(synth.gaussian(82, nv)), np.round(synth.gaussian(83, nh))
    S0, T0 = synth.spins(84, R, nv), synth.spins(85, R, nh)
    T = synth.geometric_schedule(3.0, 0.5, nsteps)
    for rule in (0, 1):
        gen = synth.logistic if rule == 0 else synth.exponential
        Fv, Fh = gen(86, (R, nsteps, nv), 1), gen(86, (R, nsteps, nh), 2)
        e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, L.PREC_BF16X1), R)
        e.set_spins(S0)
        e.set_hidden(T0)
        E = e.bip_run(rule, nsteps, Fv=Fv, Fh=Fh, fluct_per_replica=True, T=T, trace_every=2)
        S, Tm = e.get_spins(), e.get_hidden()
        for r in range(R):
            s, t, Eo = orc.bip_run(rule, W, h, b, S0[r], T0[r], nsteps, Fv[r], Fh[r], T, want_E=True)
            assert np.array_equal(s, S[r]) and np.array_equal(t, Tm[r])
            assert _close(E[:, r], Eo[1::2])


def test_bip_tc_philox_matches_f64_path(ctx, synth):
    """ISB_FLUCT_PHILOX draws the same Philox words on both paths; the tensor-core path turns them into
    decisions in fp32.  With integer couplings and T = 0 the noise drops out and both paths must agree
    exactly; at T > 0 they may differ only on rare near ties, so the energy distributions must agree."""
    L = _lib()
    nv, nh, R = 192, 128, 512
    W = np.round(synth.gaussian(91, nv * nh).reshape(nv, nh) * 1.5)
    h, b = np.round(synth.gaussian(92, nv)), np.round(synth.gaussian(93, nh))
    S0, T0 = synth.spins(94, R, nv), synth.spins(95, R, nh)
    out = {}
    for prec in (L.PREC_F64, L.PREC_BF16X1):
        e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, prec), R)
        e.set_spins(S0)
        e.set_hidden(T0)
        e.bip_run(0, 3, seed=5, T=np.zeros(3))
        out[prec] = (e.get_spins(), e.get_hidden())
    assert np.array_equal(out[L.PREC_F64][0], out[L.PREC_BF16X1][0])
    assert np.array_equal(out[L.PREC_F64][1], out[L.PREC_BF16X1][1])
    W, h, b = synth.bipartite_W(nv, nh, 96, 0.1)
    En = {}
    for prec in (L.PREC_F64, L.PREC_BF16X3):
        e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, prec), R)
        e.set_spins(S0)
        e.set_hidden(T0)
        e.bip_run(0, 30, seed=6, T=np.full(30, 1.0))
        En[prec] = e.energy()
    a, c = En[L.PREC_F64], En[L.PREC_BF16X3]
    # same noise words -> almost every chain follows the identical trajectory
    assert np.mean(np.abs(a - c) < 1e-9 * np.maximum(1, np.abs(a))) > 0.9
    assert abs(a.mean() - c.mean()) < 4 * a.std() / np.sqrt(R)


def test_bip_tc_fp16_terms(ctx, synth, monkeypatch):
    """ISB_PREC_FP16X2 / _FP16X1: fp16 terms of the power-of-two pre-scaled couplings.  Integer W is exact in one fp16
    term, so the trajectory must equal the Float64 path's bit for bit (T = 0 and caller-supplied noise, both launch
    modes); for Gaussian W the two-term split represents W to 2^-24 of max|W| (as good as W
    rounded to float), so with the same noise words almost every chain follows the Float64 trajectory, exactly as
    with three bf16 terms."""
    L = _lib()
    nv, nh, R = 192, 128, 512
    W = np.round(synth.gaussian(121, nv * nh).reshape(nv, nh) * 1.5)
    h, b = np.round(synth.gaussian(122, nv)), np.round(synth.gaussian(123, nh))
    S0, T0 = synth.spins(124, R, nv), synth.spins(125, R, nh)
    Fv, Fh = synth.logistic(126, (3, nv), 1), synth.logistic(126, (3, nh), 2)
    ref = {}
    for kw_name, kw in (("T0", dict(seed=5, T=np.zeros(3))), ("ext", dict(Fv=Fv, Fh=Fh, T=np.array([2.0, 1.0, 0.5])))):
        e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, L.PREC_F64), R)
        e.set_spins(S0)
        e.set_hidden(T0)
        e.bip_run(0, 3, **kw)
        ref[kw_name] = (e.get_spins(), e.get_hidden())
        for prec in (L.PREC_FP16X1, L.PREC_FP16X2):
            for persist in ("0", "1"):
                monkeypatch.setenv("ISB_TC_PERSIST", persist)
                e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, prec), R)
                e.set_spins(S0)
                e.set_hidden(T0)
                e.bip_run(0, 3, **kw)
                assert np.array_equal(e.get_spins(), ref[kw_name][0]), (kw_name, prec, persist)
                assert np.array_equal(e.get_hidden(), ref[kw_name][1]), (kw_name, prec, persist)
    monkeypatch.delenv("ISB_TC_PERSIST")
    W, h, b = synth.bipartite_W(nv, nh, 127, 0.1)
    En = {}
    for prec in (L.PREC_F64, L.PREC_FP16X2, L.PREC_BF16X3):
        e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, prec), R)
        e.set_spins(S0)
        e.set_hidden(T0)
        e.bip_run(0, 30, seed=6, T=np.full(30, 1.0))
        En[prec] = e.energy()
    a = En[L.PREC_F64]
    for prec in (L.PREC_FP16X2, L.PREC_BF16X3):
        c = En[prec]
        assert np.mean(np.abs(a - c) < 1e-9 * np.maximum(1, np.abs(a))) > 0.9, prec
        assert abs(a.mean() - c.mean()) < 4 * a.std() / np.sqrt(R)
    # a row-sharded model ships bf16 terms only
    with pytest.raises(L.IsbError):
        L.Model.shard_sk(ctx, 256, 2, 0, 1, 1.0, prec=L.PREC_FP16X2)


@pytest.mark.parametrize("R,nv,nh", [(300, 160, 96), (19500, 96, 80), (1000, 784, 512), (130, 784, 512), (1, 24, 17)])
def test_bip_tc_chain_resident_equals_per_half_step_launches(ctx, synth, monkeypatch, R, nv, nh):
    """The chain-resident persistent kernel (one launch for all steps, each CTA keeps its replicas) must give
    exactly what the one-launch-per-half-step path gives: same tiles, same K order, same noise words.  R = 130 / R = 1
    leave the second CTA of a pair (almost) without replicas."""
    L = _lib()
    W, h, b = synth.bipartite_W(nv, nh, 101, 0.2)
    S0, T0 = synth.spins(102, R, nv), synth.spins(103, R, nh)
    nsteps = 5
    T = synth.geometric_schedule(1.5, 0.4, nsteps)
    for rule in (0, 1):
        res = []
        for persist in ("0", "1"):
            monkeypatch.setenv("ISB_TC_PERSIST", persist)
            e = L.Ensemble(L.Model.bipartite(ctx, W, h, b, L.PREC_BF16X3), R)
            e.set_spins(S0)
            e.set_hidden(T0)
            E = e.bip_run(rule, nsteps, seed=42, step_offset=7, T=T, trace_every=2)
            res.append((e.get_spins(), e.get_hidden(), E, e.last_stats()["launches"]))
        half_steps, resident = res
        assert np.array_equal(half_steps[0], resident[0]) and np.array_equal(half_steps[1], resident[1])
        assert np.array_equal(half_steps[2], resident[2])
        assert resident[3] < half_steps[3]  # fewer launches in chain-resident mode
    # caller-supplied fluctuations through the chain-resident kernel vs the oracle-checked exact path at T = 0
    monkeypatch.setenv("ISB_TC_PERSIST", "1")
    if R <= 1000:
        Wi = np.round(W * 10.0)
        gen = synth.logistic
        Fv, Fh = gen(104, (3, nv), 1), gen(104, (3, nh), 2)
        out = []
        for prec in (L.PREC_F64, L.PREC_BF16X1):
            e = L.Ensemble(L.Model.bipartite(ctx, Wi, np.round(h * 10), np.round(b * 10), prec), R)
            e.set_spins(S0)
            e.set_hidden(T0)
            e.bip_run(0, 3, Fv=Fv, Fh=Fh, T=np.array([2.0, 1.0, 0.5]))
            out.append((e.get_spins(), e.get_hidden()))
        assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


@pytest.mark.parametrize("R,nv,nh", [(300, 160, 96), (130, 784, 512), (1, 24, 17), (19500, 96, 80)])
def test_bip_tc_cta_pairs_equal_f64_path(ctx, synth, monkeypatch, R, nv, nh):
    """The tensor-core kernel runs in CTA pairs (cta_group::2: two CTAs share one M = 256 MMA, each loads half of the
    coupling tile).  Integer couplings are exact in bf16 terms and on the int8 grid, so the pair kernel must reproduce
    the Float64 path bit for bit in spins, hidden layer and traced energies: in both launch modes, for both rules, with
    caller-supplied noise at T > 0 and with in-kernel Philox noise at T = 0 (where the noise drops out).  R = 130 / R = 1
    leave the second CTA of a pair (almost) without replicas."""
    L = _lib()
    W = np.round(synth.gaussian(111, nv * nh).reshape(nv, nh) * 1.5)
    h, b = np.round(synth.gaussian(115, nv)), np.round(synth.gaussian(116, nh))
    S0, T0 = synth.spins(112, R, nv), synth.spins(113, R, nh)
    nsteps = 4
    Fv, Fh = synth.logistic(114, (nsteps, nv), 1), synth.logistic(114, (nsteps, nh), 2)
    runs = (dict(Fv=Fv, Fh=Fh, T=synth.geometric_schedule(1.5, 0.4, nsteps)),
            dict(seed=42, step_offset=7, T=np.zeros(nsteps)))

    def run(m, rule, kw):
        e = L.Ensemble(m, R)
        e.set_spins(S0)
        e.set_hidden(T0)
        E = e.bip_run(rule, nsteps, trace_every=2, **kw)
        return e.get_spins(), e.get_hidden(), E

    ref_model = L.Model.bipartite(ctx, W, h, b, L.PREC_F64)
    models = {prec: L.Model.bipartite(ctx, W, h, b, prec) for prec in (L.PREC_BF16X3, L.PREC_BF16X1, L.PREC_I8X3)}
    for m in models.values():
        assert np.array_equal(m.effective_couplings(), W)
    for rule in (0, 1):
        for i, kw in enumerate(runs):
            ref = run(ref_model, rule, kw)
            for prec, m in models.items():
                for persist in ("0", "1"):
                    monkeypatch.setenv("ISB_TC_PERSIST", persist)
                    S, Tm, E = run(m, rule, kw)
                    assert np.array_equal(S, ref[0]) and np.array_equal(Tm, ref[1]), (rule, i, prec, persist)
                    assert np.array_equal(E, ref[2]), (rule, i, prec, persist)


# ---------------------------------------------------------------- edge cases
def test_edge_cases(ctx, orc, synth):
    L = _lib()
    N, R = 40, 3
    J, h = synth.sk_J(N, 1), synth.gaussian(2, N) * 0.1
    S0 = synth.spins(3, R, N)
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    # zero steps: nothing happens, flips are zero
    out = e.ssf_run(1, 0, T=np.ones(1))
    assert np.array_equal(e.get_spins(), S0) and out["flips"].tolist() == [0, 0, 0]
    # trace stride longer than the run: no trace rows
    out = e.ssf_run(1, 5, fluct=np.zeros(5), T=np.ones(5), trace_every=100)
    assert out["E"] is None
    # T = 0 (the annealing end point): deterministic quench, ties give +1; negative T is accepted like the reference
    e.set_spins(S0)
    e.ssf_run(2, 3 * N, fluct=synth.exponential(4, 3 * N), T=np.zeros(1), steps_per_T=3 * N)
    s, *_ = orc.ssf_run(2, J, h, S0[0], 3 * N, fluct=synth.exponential(4, 3 * N), T=np.zeros(1), steps_per_T=3 * N)
    assert np.array_equal(e.get_spins()[0], s)
    e.set_spins(S0)
    e.ssf_run(1, N, fluct=synth.logistic(5, N), T=np.array([-0.5]), steps_per_T=N)
    s, *_ = orc.ssf_run(1, J, h, S0[1], N, fluct=synth.logistic(5, N), T=np.array([-0.5]), steps_per_T=N)
    assert np.array_equal(e.get_spins()[1], s)
    # a site list that hammers one site, and a sweep starting at the last site
    e.set_spins(S0)
    nodes = np.array([7] * 20 + [0, 39] * 5, dtype=np.int32)
    fl = synth.logistic(6, 30)
    e.ssf_run(1, 30, nodes=nodes, fluct=fl, T=np.full(30, 1.3))
    s, *_ = orc.ssf_run(1, J, h, S0[2], 30, nodes=nodes, fluct=fl, T=np.full(30, 1.3))
    assert np.array_equal(e.get_spins()[2], s)
    e.set_spins(S0)
    e.ssf_run(2, 2 * N + 1, start=N - 1, fluct=synth.exponential(7, 2 * N + 1), T=np.array([0.9]), steps_per_T=2 * N + 1)
    s, *_ = orc.ssf_run(2, J, h, S0[0], 2 * N + 1, start=N - 1, fluct=synth.exponential(7, 2 * N + 1), T=np.array([0.9]),
                        steps_per_T=2 * N + 1)
    assert np.array_equal(e.get_spins()[0], s)
    # one isolated spin in a field, one replica
    e1 = L.Ensemble(L.Model.dense(ctx, np.zeros((1, 1)), np.array([0.3]), L.PREC_F64), 1)
    e1.set_spins(np.array([[-1]], dtype=np.int8))
    e1.ssf_run(0, 1)
    assert e1.get_spins()[0, 0] == -1  # Hopfield: J.s - h = -0.3 < 0 (the minus-h quirk, SingleSpinFlip.jl:33-34)
    e1.ssf_run(1, 1, fluct=np.zeros(1), T=np.ones(1))
    assert e1.get_spins()[0, 0] == 1


def test_many_replicas_more_than_two_waves(ctx, orc, synth):
    """R far above chains-per-CTA x SMs (several waves of CTAs), checked on a sample of replicas."""
    L = _lib()
    N, R, nsteps = 96, 9000, 96 * 4
    J, h = synth.sk_J(N, 9), np.zeros(N)
    S0 = synth.spins(10, R, N)
    T = np.array([1.2, 0.8, 0.5, 0.3])
    e = L.Ensemble(L.Model.dense(ctx, J, h, L.PREC_F64), R)
    e.set_spins(S0)
    e.ssf_run(1, nsteps, seed=77, T=T, steps_per_T=N)
    S = e.get_spins()
    for r in (0, 1, 4499, 8998, 8999):
        fl = ctx.philox_fluct(1, 77, 0, r, 1, nsteps)[0]
        s, *_ = orc.ssf_run(1, J, h, S0[r], nsteps, fluct=fl, T=T, steps_per_T=N)
        assert np.array_equal(s, S[r])


@pytest.mark.parametrize("hmag", [0.05, 0.0])
@pytest.mark.parametrize("path", ["dense", "sparse"])
def test_long_run_with_commensurate_couplings_at_zero_temperature(ctx, orc, synth, path, hmag):
    """Couplings +-0.1 / +-0.3 (sums that round, exact cancellations; with h = 0 the reference's field is an exact or
    one-ulp tie again and again): the reference recomputes a fresh row dot at every step (src/SpinSystems.jl:80-83), the
    kernels maintain the field incrementally.  For such couplings (a small non-dyadic alphabet) the kernels run with the
    near-tie guard: a decision within 2^-30 of the field scale is taken on a fresh sequential row dot, and the cached
    fields are refreshed every ISB_FIELD_REFRESH_SWEEPS sweeps.  300 sweeps of T = 0 dynamics in runs of 75 sweeps
    must follow the oracle bit for bit."""
    import scipy.sparse as sp
    L = _lib()
    n, R, sweeps, per = 96, 12, 300, 75
    g = synth.gaussian(91, n * n).reshape(n, n)
    J = np.where(g > 0.8, 0.3, np.where(g > 0.0, 0.1, np.where(g > -0.8, -0.1, -0.3)))
    J = np.where(np.abs(synth.gaussian(92, n * n).reshape(n, n)) < 0.25, J, 0.0)   # ~20 % of the pairs: even degrees occur
    J = np.triu(J, 1)
    J = J + J.T
    h = np.where(synth.gaussian(93, n) > 0, hmag, -hmag)      # hmag = 0.05 breaks the exact zero-field ties, 0 keeps them
    S0 = synth.spins(94, R, n)
    m = L.Model.sparse(ctx, sp.csc_matrix(J), h) if path == "sparse" else L.Model.dense(ctx, J, h, L.PREC_F64)
    e = L.Ensemble(m, R)
    e.set_spins(S0)
    e.set_tie_eps(1e-12)
    ties = 0
    for c in range(sweeps // per):
        e.ssf_run(L.RULE_GLAUBER, per * n, fluct=np.zeros(per * n), T=np.zeros(1), steps_per_T=per * n)
        ties += e.last_stats()["near_ties"]
    S = e.get_spins()
    bad = 0
    for r in range(R):
        s, *_ = orc.ssf_run(orc.GLAUBER, J, h, S0[r], sweeps * n, fluct=np.zeros(sweeps * n), T=np.zeros(1), steps_per_T=sweeps * n)
        bad += int(not np.array_equal(s, S[r]))
    print(f"\n[{path}, |h| = {hmag}] commensurate couplings, T = 0, {sweeps} sweeps: {bad} of {R} chains differ, {ties} near-tie decisions audited")
    assert bad == 0, "a decision differs from the reference's fresh row dot"
